// Discriminative loss, forward and backward, as segmented reductions over the
// embedding map.  Replaces the broadcast-and-reduce PyTorch graph of
//   /root/reference/code/lib/losses/discriminative.py:7-62   (calculate_means)
//   /root/reference/code/lib/losses/discriminative.py:65-95  (calculate_variance_term, else-branch)
//   /root/reference/code/lib/losses/discriminative.py:98-132 (calculate_distance_term)
//   /root/reference/code/lib/losses/discriminative.py:135-147 (calculate_regularization_term)
//   /root/reference/code/lib/losses/discriminative.py:149-160 (calculate_q_regularization_term)
//   /root/reference/code/lib/losses/discriminative.py:162-188 (discriminative_loss composite)
//
// Data layout in HBM: emb is the network's NCHW map [bs][C][H*W] (pixel index
// contiguous), so a warp reads 32 consecutive pixels of one channel per load
// (128 B, fully coalesced) and each thread keeps the C channel values of its
// pixel in registers.  The target is read as handed over: a u8 label map
// [bs][H*W] (255 = background) or the reference's dense one-hot/float mask
// [bs][K][H*W] (f32 / i64 / u8).
//
// Forward = one cooperative kernel.  Each image is owned by G co-resident CTAs.
//   phase 1: per-instance sums  s_k = sum_p m_pk x_p, counts, q-regulariser
//   -- per-image barrier (all partial sums are in L2) --
//   phase 2: means -> smem, hinge sum  sum_p m_pk max(|x_p-mu_k|-dv,0)^2 and the
//            per-instance hinge-gradient sums A_k kept for backward; the second
//            read of the image comes out of L2, not HBM.
// A thread walks DOWN a pixel column: instance masks are spatially coherent, so
// the running (label, partial sum) pair stays in registers until the label
// changes and only then is flushed with fire-and-forget float REDs.
//
// Backward = a tiny per-image prep kernel (normalised-mean Jacobian, distance /
// regulariser gradients on the K x C means) + one streaming pass that reads the
// embedding and target once and writes grad_emb once.
#include "isa_common.cuh"
#include <math.h>

namespace {

enum { TGT_LABEL_U8 = 0, TGT_DENSE_F32 = 1, TGT_DENSE_I64 = 2, TGT_DENSE_U8 = 3 };
enum { ROUTE_LAB = 0, ROUTE_COL_THEN_LAB = 1, ROUTE_COL = 2 };   // ISA_DISC_ROUTE_* of include/isa_b200.h

constexpr int kThreads = 256;
constexpr int kWarps = kThreads / 32;
constexpr int kLabMaxCtas = 640;     // upper bound of the label-map forward's grid (2 CTAs per SM on any sm_100 part)

struct DiscWs {
  // zeroed region
  float* sums;        // [bs][K][C+1], last column = count
  float* gsum;        // [bs][K][C]    A_k = sum_p m_pk * dh^2/dx
  float* var_sum;     // [bs]
  double* qsum;       // [1]
  double* nfg;        // [1]
  unsigned* img_cnt;  // [bs]
  unsigned* done_cnt; // [1]
  int* not_onehot;    // [1] dense target only: some pixel has several / non-unit entries -> keep the dense path
  unsigned* tick1;    // [bs] label-map forward: CTAs of the image that have written their phase-1 partials
  unsigned* tick2;    // [bs] ... phase-2 partials
  unsigned* lab_bar;  // [1]  its grid barrier
  // not zeroed
  unsigned char* labels;  // [bs][P] u8 label map distilled from a dense one-hot target (255 = background)
  float* rnorm;   // [bs][K]  |mu~_k| before normalisation
  float* Nb;      // [bs]
  float* dist_b;  // [bs]
  float* reg_b;   // [bs]
  float* T;       // [bs][K][C]  bwd: dL/d(mu~_k) / count_k
  float* coef;    // [bs] cdir_b, then [1] cq
  float* part;    // [kLabMaxCtas][K][C+1] per-CTA partial sums of the label-map forward (phase 1, then phase 2)
  double* partq;  // [kLabMaxCtas][3]      per-CTA q-regulariser sum, foreground count, hinge sum
  double* qb;     // [bs][2]               per-image q-regulariser sum and foreground count (fixed-order folds)
  size_t zero_bytes;
  size_t total_bytes;
};

static DiscWs carve(void* base, int bs, int C, int K, int P) {
  DiscWs w;
  char* p = (char*)base;
  size_t off = 0;
  auto take = [&](size_t bytes) {
    char* r = p ? p + off : nullptr;
    off += isa_align_up(bytes, 16);
    return r;
  };
  w.qsum = (double*)take(sizeof(double));
  w.nfg = (double*)take(sizeof(double));
  w.sums = (float*)take(sizeof(float) * (size_t)bs * K * (C + 1));
  w.gsum = (float*)take(sizeof(float) * (size_t)bs * K * C);
  w.var_sum = (float*)take(sizeof(float) * bs);
  w.img_cnt = (unsigned*)take(sizeof(unsigned) * bs);
  w.done_cnt = (unsigned*)take(sizeof(unsigned));
  w.not_onehot = (int*)take(sizeof(int));
  w.tick1 = (unsigned*)take(sizeof(unsigned) * bs);
  w.tick2 = (unsigned*)take(sizeof(unsigned) * bs);
  w.lab_bar = (unsigned*)take(sizeof(unsigned));
  w.zero_bytes = off;
  w.labels = (unsigned char*)take((size_t)bs * P);
  w.rnorm = (float*)take(sizeof(float) * (size_t)bs * K);
  w.Nb = (float*)take(sizeof(float) * bs);
  w.dist_b = (float*)take(sizeof(float) * bs);
  w.reg_b = (float*)take(sizeof(float) * bs);
  w.T = (float*)take(sizeof(float) * (size_t)bs * K * C);
  w.coef = (float*)take(sizeof(float) * (bs + 1));
  w.part = (float*)take(sizeof(float) * (size_t)kLabMaxCtas * K * (C + 1));
  w.partq = (double*)take(sizeof(double) * (size_t)kLabMaxCtas * 3);
  w.qb = (double*)take(sizeof(double) * (size_t)bs * 2);
  w.total_bytes = off;
  return w;
}

struct FwdParams {
  const float* emb;
  const void* target;
  const int* n_objects;
  int target_kind;
  int bs, C, H, W, K;
  float delta_v, delta_d;
  int norm;
  int normalize_means;
  float w_var, w_dist, w_reg, w_q;
  DiscWs ws;
  float* out_loss;   // [1]
  float* out_terms;  // [4] var, dist, reg, qreg (unweighted)
  float* out_means;  // [bs][K][C]
  const float* q_den;  // optional override of the q-regulariser denominator (data parallel), else null
  int G;             // CTAs per image (1 => CTA loops over images, no inter-CTA barrier)
  int strips, rowsplits, rpt;
  int lab_kernel_follows;   // dense target: skip the work when the masks turn out one-hot (the label-map kernel runs next)
};

// Reads the (up to K) mask weights of pixel p.  Returns the number of non-zero
// entries; k1/w1 = the first one; fg = sum over all K channels
// (discriminative.py:151 sums the target over every instance channel).
template <int KIND>
__device__ __forceinline__ int read_mask(const void* __restrict__ tgt, size_t img_off_px, int p, int P, int K,
                                         int& k1, float& w1, float& fg) {
  if (KIND == TGT_LABEL_U8) {
    const unsigned char l = __ldg((const unsigned char*)tgt + img_off_px + p);
    if ((int)l < K) { k1 = l; w1 = 1.f; fg = 1.f; return 1; }
    k1 = -1; w1 = 0.f; fg = 0.f; return 0;
  } else {
    int nnz = 0; k1 = -1; w1 = 0.f; fg = 0.f;
    for (int k = 0; k < K; ++k) {
      float m;
      const size_t idx = (img_off_px * (size_t)K) + (size_t)k * P + p;
      if (KIND == TGT_DENSE_F32) m = __ldg((const float*)tgt + idx);
      else if (KIND == TGT_DENSE_I64) m = (float)__ldg((const long long*)tgt + idx);
      else m = (float)__ldg((const unsigned char*)tgt + idx);
      if (m != 0.f) { fg += m; if (nnz == 0) { k1 = k; w1 = m; } ++nnz; }
    }
    return nnz;
  }
}
template <int KIND>
__device__ __forceinline__ float read_mask_k(const void* __restrict__ tgt, size_t img_off_px, int p, int P, int K, int k) {
  const size_t idx = (img_off_px * (size_t)K) + (size_t)k * P + p;
  if (KIND == TGT_DENSE_F32) return __ldg((const float*)tgt + idx);
  if (KIND == TGT_DENSE_I64) return (float)__ldg((const long long*)tgt + idx);
  if (KIND == TGT_DENSE_U8) return (float)__ldg((const unsigned char*)tgt + idx);
  return 0.f;
}

// Warp-cooperative flush of the lanes' running (label, partial sums) into the CTA's shared accumulators.
// Every lane parks its `width` partials in the warp's slab (row stride width | 1: conflict free); then, for each
// distinct label held in the warp, lane c sums column c over the lanes holding that label and issues ONE shared
// atomic -- instead of 32 lanes x width same-address atomics (which serialise 32-way and made the first
// shared-memory version slower than flushing to L2).  Must be called by all 32 lanes.
template <int CP>
__device__ __forceinline__ void warp_flush(float* __restrict__ slab, float* __restrict__ dst, int dst_stride, int width, int cur,
                                           const float (&acc)[CP], float cnt, int C) {
  const int lane = threadIdx.x & 31;
  const int SS = width | 1;
  unsigned rem = __ballot_sync(0xffffffffu, cur >= 0);
  if (rem == 0) return;
#pragma unroll
  for (int c = 0; c < CP; ++c)
    if (c < C) slab[lane * SS + c] = acc[c];
  if (width > C) slab[lane * SS + C] = cnt;
  __syncwarp();
  while (rem) {
    const int leader = __ffs(rem) - 1;
    const int L = __shfl_sync(0xffffffffu, cur, leader);
    const unsigned grp = __ballot_sync(0xffffffffu, cur == L);
    for (int col = lane; col < width; col += 32) {
      float t = 0.f;
      unsigned g = grp;
      while (g) {
        const int r = __ffs(g) - 1;
        g &= g - 1;
        t += slab[r * SS + col];
      }
      if (t != 0.f) atomicAdd(dst + (size_t)L * dst_stride + col, t);
    }
    rem &= ~grp;
  }
  __syncwarp();
}

// hinge on one (pixel, instance) pair: returns w*h^2 and the gradient scale so
// that d(w h^2)/dx_c = gs * dir_c, dir_c = (x_c-mu_c) for L2, sign(x_c-mu_c) for L1.
template <int CP>
__device__ __forceinline__ float hinge_pair(const float (&x)[CP], const float* __restrict__ mu, int C, int norm, float delta_v, float w,
                                            float (&dir)[CP], float& gs) {
  float d = 0.f;
  if (norm == 2) {
#pragma unroll
    for (int c = 0; c < CP; ++c)
      if (c < C) { dir[c] = x[c] - mu[c]; d = fmaf(dir[c], dir[c], d); }
    d = sqrtf(d);
  } else {
#pragma unroll
    for (int c = 0; c < CP; ++c)
      if (c < C) { const float t = x[c] - mu[c]; d += fabsf(t); dir[c] = (t > 0.f) ? 1.f : ((t < 0.f) ? -1.f : 0.f); }
  }
  const float h = fmaxf(d - delta_v, 0.f);
  if (norm == 2) gs = (h > 0.f && d > 0.f) ? 2.f * w * h / d : 0.f;
  else gs = (h > 0.f) ? 2.f * w * h : 0.f;
  return w * h * h;
}

template <int CP, int KIND>
__device__ __forceinline__ void disc_fwd_body(const FwdParams& prm, const void* __restrict__ target) {
  extern __shared__ float smem[];  // means [K][CP+1] | CTA-level sums [K][C+1] | CTA-level hinge-gradient sums [K][C]
  __shared__ float s_red[kWarps];
  __shared__ int s_flag;
  const int C = prm.C, K = prm.K, W = prm.W, H = prm.H, P = H * W;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int MS = CP + 1;
  float* __restrict__ s_sum = smem + K * MS;            // [K][C+1]
  float* __restrict__ s_gs = s_sum + K * (C + 1);       // [K][C]
  float* __restrict__ slab = s_gs + K * C + warp * 32 * ((C + 1) | 1);   // per-warp [32][(C+1)|1] staging for warp_flush

  const int G = prm.G;
  const int b0 = blockIdx.x / G, g = blockIdx.x % G;
  const int img_step = gridDim.x / G;
  const int tiles = prm.strips * prm.rowsplits;
  const int warps_per_img = G * kWarps;

  double q_acc = 0.0, nfg_acc = 0.0;
  int round = 0;
  for (int b = b0; b < prm.bs; b += img_step, ++round) {
    const int nb = min(max(__ldg(prm.n_objects + b), 0), K);
    const float* __restrict__ emb = prm.emb + (size_t)b * C * P;
    const size_t img_off_px = (size_t)b * P;
    float* __restrict__ sums = prm.ws.sums + (size_t)b * K * (C + 1);
    for (int i = threadIdx.x; i < K * (2 * C + 1); i += kThreads) s_sum[i] = 0.f;   // s_sum and s_gs are adjacent
    __syncthreads();

    // ---------------- phase 1: per-instance sums, counts, q-regulariser ----------------
    // runs are flushed to the CTA's shared-memory accumulators (native fp32 shared atomics); the CTA then adds
    // its non-zero entries to the image's sums in L2 once -- r1a's version flushed every run straight to L2 and
    // spent a third of the kernel waiting at the per-image barrier for those float atomics to drain
    for (int t = g * kWarps + warp; t < tiles; t += warps_per_img) {
      const int strip = t % prm.strips, rs = t / prm.strips;
      const int xcol = strip * 32 + lane;
      const int y0 = rs * prm.rpt, y1 = min(H, y0 + prm.rpt);
      const bool live = xcol < W;                       // dead lanes still take part in the warp-wide flushes
      float acc[CP];
#pragma unroll
      for (int c = 0; c < CP; ++c) acc[c] = 0.f;
      float cnt = 0.f;
      float q_tile = 0.f, nfg_tile = 0.f;
      int cur = -1;
#pragma unroll 2
      for (int y = y0; y < y1; ++y) {
        const int p = y * W + xcol;
        int k1 = -1; float w1 = 0.f, fg = 0.f;
        int nnz = 0;
        float x[CP];
        if (live) {
          nnz = read_mask<KIND>(target, img_off_px, p, P, K, k1, w1, fg);
#pragma unroll
          for (int c = 0; c < CP; ++c) x[c] = (c < C) ? __ldg(emb + (size_t)c * P + p) : 0.f;
          // q-regulariser: (|x*fg|_2 - 1)^2 for EVERY pixel (background adds 1).
          float ss = 0.f;
#pragma unroll
          for (int c = 0; c < CP; ++c) { const float tq = x[c] * fg; ss = fmaf(tq, tq, ss); }
          const float l2 = sqrtf(ss);
          q_tile += (l2 - 1.f) * (l2 - 1.f);
          nfg_tile += fg;
        }
        const bool single = (nnz == 1) && (k1 < nb);
        // a lane whose run ends makes the whole warp flush (lanes in the middle of a run simply restart it);
        // measured faster than letting that lane issue its C+1 shared atomics alone (146 vs 171 us at bs 16, 256^2)
        if (__any_sync(0xffffffffu, single && cur >= 0 && k1 != cur)) {
          warp_flush<CP>(slab, s_sum, C + 1, C + 1, cur, acc, cnt, C);
#pragma unroll
          for (int c = 0; c < CP; ++c) acc[c] = 0.f;
          cnt = 0.f; cur = -1;
        }
        if (single) {
          cur = k1;
#pragma unroll
          for (int c = 0; c < CP; ++c) acc[c] = fmaf(w1, x[c], acc[c]);
          cnt += w1;
        } else if (nnz > 1) {
          // soft / overlapping masks: every non-zero entry goes straight to the shared accumulators.
          for (int k = k1; k < nb; ++k) {
            const float m = read_mask_k<KIND>(target, img_off_px, p, P, K, k);
            if (m != 0.f) {
              float* row = s_sum + k * (C + 1);
#pragma unroll
              for (int c = 0; c < CP; ++c) if (c < C) atomicAdd(row + c, m * x[c]);
              atomicAdd(row + C, m);
            }
          }
        }
      }
      warp_flush<CP>(slab, s_sum, C + 1, C + 1, cur, acc, cnt, C);
      q_acc += (double)q_tile;
      nfg_acc += (double)nfg_tile;
    }
    __syncthreads();
    for (int i = threadIdx.x; i < K * (C + 1); i += kThreads) {
      const float v = s_sum[i];
      if (v != 0.f) atomicAdd(sums + i, v);
    }

    // ---------------- per-image barrier ----------------
    if (G > 1) {
      group_barrier(prm.ws.img_cnt + b, (unsigned)G);
    } else {
      __threadfence();
      __syncthreads();
    }

    // ---------------- means -> smem ----------------
    for (int k = warp; k < K; k += kWarps) {
      float v = 0.f;
      float cntk = 0.f;
      if (k < nb) {
        cntk = __ldcg(sums + (size_t)k * (C + 1) + C);
        if (lane < C) v = __ldcg(sums + (size_t)k * (C + 1) + lane) / cntk;
        // CP may exceed 32 (CP=64): second half handled below
      }
      float v2 = 0.f;
      if (CP > 32 && k < nb && lane + 32 < C) v2 = __ldcg(sums + (size_t)k * (C + 1) + lane + 32) / cntk;
      float r = 1.f;
      if (k < nb) {
        const float n2 = warp_sum(v * v + v2 * v2);
        r = sqrtf(n2);
        if (prm.normalize_means) { v = v / r; v2 = v2 / r; }
      }
      if (lane < CP) smem[k * MS + lane] = v;
      if (CP > 32 && lane + 32 < CP) smem[k * MS + lane + 32] = v2;
      if (g == 0) {
        if (lane < C) prm.out_means[((size_t)b * K + k) * C + lane] = v;
        if (CP > 32 && lane + 32 < C) prm.out_means[((size_t)b * K + k) * C + lane + 32] = v2;
        if (lane == 0) prm.ws.rnorm[(size_t)b * K + k] = r;
      }
    }
    __syncthreads();

    if (g == 0) {
      // N_b, distance term and regulariser of this image (K^2*C work, one CTA).
      float nsum = 0.f;
      for (int k = threadIdx.x; k < nb; k += kThreads) {
        const float ck = __ldcg(sums + (size_t)k * (C + 1) + C);
        // an instance id below n_objects with no pixels makes the reference's
        // mean 0/0 and its whole loss NaN (discriminative.py:41-42,84-85)
        nsum += (ck == 0.f) ? nanf("") : ck;
      }
      float dsum = 0.f, rsum = 0.f;
      if (prm.w_dist != 0.f && nb > 1) {
        for (int ij = threadIdx.x; ij < nb * nb; ij += kThreads) {
          const int i = ij / nb, j = ij % nb;
          if (i == j) continue;
          float e = 0.f;
          for (int c = 0; c < C; ++c) {
            const float t = smem[i * MS + c] - smem[j * MS + c];
            e = (prm.norm == 2) ? fmaf(t, t, e) : e + fabsf(t);
          }
          if (prm.norm == 2) e = sqrtf(e);
          const float m = fmaxf(2.f * prm.delta_d - e, 0.f);
          dsum = fmaf(m, m, dsum);
        }
      }
      if (prm.w_reg != 0.f) {
        for (int k = threadIdx.x; k < nb; k += kThreads) {
          float e = 0.f;
          for (int c = 0; c < C; ++c) {
            const float t = smem[k * MS + c];
            e = (prm.norm == 2) ? fmaf(t, t, e) : e + fabsf(t);
          }
          rsum += (prm.norm == 2) ? sqrtf(e) : e;
        }
      }
      nsum = warp_sum(nsum); dsum = warp_sum(dsum); rsum = warp_sum(rsum);
      __shared__ float s3[3][kWarps];
      if (lane == 0) { s3[0][warp] = nsum; s3[1][warp] = dsum; s3[2][warp] = rsum; }
      __syncthreads();
      if (threadIdx.x == 0) {
        float a = 0.f, d = 0.f, r = 0.f;
        for (int w = 0; w < kWarps; ++w) { a += s3[0][w]; d += s3[1][w]; r += s3[2][w]; }
        prm.ws.Nb[b] = a;
        prm.ws.dist_b[b] = (nb > 1) ? d / (float)(nb * (nb - 1)) : 0.f;
        prm.ws.reg_b[b] = r / (float)nb;  // torch.mean over an empty slice is nan, as 0/0 here
      }
    }

    // ---------------- phase 2: hinge sum + per-instance hinge-gradient sums ----------------
    float var_acc = 0.f;
    float* __restrict__ gsum = prm.ws.gsum + (size_t)b * K * C;
    for (int t = g * kWarps + warp; t < tiles; t += warps_per_img) {
      const int strip = t % prm.strips, rs = t / prm.strips;
      const int xcol = strip * 32 + lane;
      const int y0 = rs * prm.rpt, y1 = min(H, y0 + prm.rpt);
      const bool live = xcol < W;
      float acc[CP];
#pragma unroll
      for (int c = 0; c < CP; ++c) acc[c] = 0.f;
      int cur = -1;
#pragma unroll 2
      for (int y = y0; y < y1; ++y) {
        const int p = y * W + xcol;
        int k1 = -1; float w1 = 0.f, fg = 0.f;
        int nnz = 0;
        if (live) nnz = read_mask<KIND>(target, img_off_px, p, P, K, k1, w1, fg);
        const bool use = nnz > 0 && k1 < nb;
        const bool single = use && nnz == 1;
        if (__any_sync(0xffffffffu, single && cur >= 0 && k1 != cur)) {
          warp_flush<CP>(slab, s_gs, C, C, cur, acc, 0.f, C);
#pragma unroll
          for (int c = 0; c < CP; ++c) acc[c] = 0.f;
          cur = -1;
        }
        if (!use) continue;
        float x[CP];
#pragma unroll
        for (int c = 0; c < CP; ++c) x[c] = (c < C) ? __ldg(emb + (size_t)c * P + p) : 0.f;
        float dir[CP]; float gs;
        if (single) {
          var_acc += hinge_pair<CP>(x, smem + k1 * MS, C, prm.norm, prm.delta_v, w1, dir, gs);
          cur = k1;
#pragma unroll
          for (int c = 0; c < CP; ++c) if (c < C) acc[c] = fmaf(gs, dir[c], acc[c]);
        } else {
          for (int k = k1; k < nb; ++k) {
            const float m = read_mask_k<KIND>(target, img_off_px, p, P, K, k);
            if (m != 0.f) {
              var_acc += hinge_pair<CP>(x, smem + k * MS, C, prm.norm, prm.delta_v, m, dir, gs);
#pragma unroll
              for (int c = 0; c < CP; ++c) if (c < C) atomicAdd(s_gs + k * C + c, gs * dir[c]);
            }
          }
        }
      }
      warp_flush<CP>(slab, s_gs, C, C, cur, acc, 0.f, C);
    }
    var_acc = warp_sum(var_acc);
    if (lane == 0) s_red[warp] = var_acc;
    __syncthreads();
    for (int i = threadIdx.x; i < K * C; i += kThreads) {
      const float v = s_gs[i];
      if (v != 0.f) atomicAdd(gsum + i, v);
    }
    if (threadIdx.x == 0) {
      float v = 0.f;
      for (int w = 0; w < kWarps; ++w) v += s_red[w];
      atomicAdd(prm.ws.var_sum + b, v);
    }
    __syncthreads();  // smem means are reused by the next image
  }

  // ---------------- q-regulariser partials ----------------
  q_acc = warp_sum_d(q_acc);
  nfg_acc = warp_sum_d(nfg_acc);
  if (lane == 0) { atomicAdd(prm.ws.qsum, q_acc); atomicAdd(prm.ws.nfg, nfg_acc); }

  // ---------------- last CTA: combine the scalars ----------------
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) s_flag = (atomicAdd(prm.ws.done_cnt, 1u) == gridDim.x - 1);
  __syncthreads();
  if (s_flag && warp == 0) {
    __threadfence();
    float v = 0.f, d = 0.f, r = 0.f;
    for (int b = lane; b < prm.bs; b += 32) {
      v += __ldcg(prm.ws.var_sum + b) / __ldcg(prm.ws.Nb + b);
      d += __ldcg(prm.ws.dist_b + b);
      r += __ldcg(prm.ws.reg_b + b);
    }
    v = warp_sum(v); d = warp_sum(d); r = warp_sum(r);
    if (lane == 0) {
      const float inv_bs = 1.f / (float)prm.bs;
      const double qs = __ldcg(prm.ws.qsum), nf = __ldcg(prm.ws.nfg);
      // discriminative.py:153-159: num = int(sum(target)); loss = sum(...)/num
      const double qden = prm.q_den ? (double)__ldg(prm.q_den) : (double)(long long)nf;
      const float qreg = (float)(qs / qden);
      const float var_t = v * inv_bs;
      const float dist_t = (prm.w_dist != 0.f) ? d * inv_bs : 0.f;
      const float reg_t = (prm.w_reg != 0.f) ? r * inv_bs : 0.f;
      prm.out_terms[0] = var_t; prm.out_terms[1] = dist_t; prm.out_terms[2] = reg_t; prm.out_terms[3] = qreg;
      float loss = 0.f;
      if (prm.w_var != 0.f) loss += prm.w_var * var_t;
      if (prm.w_dist != 0.f) loss += prm.w_dist * dist_t;
      if (prm.w_reg != 0.f) loss += prm.w_reg * reg_t;
      if (prm.w_q != 0.f) loss += prm.w_q * qreg;
      prm.out_loss[0] = loss;
    }
  }
}

// A dense one-hot target (what the reference's collate emits: K x 4..8 bytes per pixel) is distilled once into a
// u8 label map in the workspace (onehot_to_labels_kernel); forward and backward then read 1 byte per pixel.  If any
// pixel turns out not to be one-hot (soft or overlapping masks) the flag is set and the kernels keep the dense path.
template <int CP, int KIND>
__global__ void __launch_bounds__(kThreads, (CP <= 32) ? 2 : 1) disc_fwd_kernel(const FwdParams prm) {
  if (KIND == TGT_LABEL_U8) {
    disc_fwd_body<CP, TGT_LABEL_U8>(prm, prm.target);
  } else if (__ldcg(prm.ws.not_onehot) == 0) {
    if (prm.lab_kernel_follows) return;              // one-hot after all: disc_fwd_lab_kernel (launched next) does the work
    disc_fwd_body<CP, TGT_LABEL_U8>(prm, prm.ws.labels);
  } else {
    disc_fwd_body<CP, KIND>(prm, prm.target);
  }
}


// ---------------------------------------------------------------- forward, label-map targets (the hot configuration)
// One cooperative kernel, ONE grid barrier, no float atomics (bit-reproducible run to run):
//   phase 1   every CTA owns a contiguous pixel range of one image; a warp takes 32 consecutive pixels at a time
//             (lane = pixel: C coalesced 128-byte loads, the pixel's channels stay in registers) and reduces each channel
//             over the lanes that share a label with shuffles -- instance masks are spatially coherent, so most segments
//             hold ONE label and cost 5 shuffles per channel -- into the WARP's private shared-memory accumulators;
//             warps are folded in a fixed order into the CTA's partial, the last CTA of the image (a ticket) folds the
//             image's partials in CTA order and finishes means, norms, N_b, distance and regulariser terms;
//   barrier   all images' means are in L2;
//   phase 2   the same walk (the embedding comes back from L2: 100 MB at batch 16 against 126 MB of L2): hinge, hinge sum
//             and the per-instance hinge-gradient sums kept for backward, folded the same way; the last CTA overall
//             combines the scalars.
// The previous version walked pixel columns with running (label, sum) pairs and flushed the whole warp through shared
// memory whenever ONE lane's label changed (every ~1.5 rows): 134 us at batch 16 (0.12 of the HBM roofline), 40 % of the
// samples at its per-image barriers.  Soft / overlapping masks keep that kernel (disc_fwd_kernel above).
struct LabParams {
  FwdParams f;
  int G;          // CTAs per image
  int chunk;      // pixels per CTA (multiple of 32)
  int priv;       // 1: per-warp accumulators (deterministic); 0: one CTA accumulator with shared atomics (K * C too large)
};

// Sum of every channel over the 32 lanes with 31 shuffles instead of 5 per channel (recursive halving: at each step a
// lane hands half of its remaining channels to its partner and adds the partner's half of the others).  N = channel
// count padded to a power of two (<= 32); afterwards v[0] of lane l is the total of channel (l * N) / 32.
template <int N>
__device__ __forceinline__ void warp_reduce_channels(float (&v)[N], int lane) {
  static_assert(N == 8 || N == 16 || N == 32, "pad the channel count to 8, 16 or 32");
  int o = 16;
#pragma unroll
  for (int n = N; n > 1; n >>= 1, o >>= 1) {
    const bool up = (lane & o) != 0;
#pragma unroll
    for (int i = 0; i < n / 2; ++i) {
      const float send = up ? v[i] : v[i + n / 2];
      const float keep = up ? v[i + n / 2] : v[i];
      v[i] = keep + __shfl_xor_sync(0xffffffffu, send, o);
    }
  }
#pragma unroll
  for (; o >= 1; o >>= 1) v[0] += __shfl_xor_sync(0xffffffffu, v[0], o);
}

// Running per-instance sums of one warp: lane l keeps the running total of "its" channel(s) for the warp's current label in
// registers; shared memory (the warp's private accumulators, or the CTA's with atomics) is touched only when the label
// changes -- instance masks are spatially coherent, so that is rare.
template <int CP>
struct WarpRun {
  static constexpr int N = CP <= 8 ? 8 : CP <= 16 ? 16 : 32;      // padded width of one reduction
  static constexpr int R = CP <= 32 ? 1 : 2;                      // CP = 64: two reductions of 32 channels
  float run[R];
  float cnt;
  int cur;
  __device__ __forceinline__ void init() {
#pragma unroll
    for (int r = 0; r < R; ++r) run[r] = 0.f;
    cnt = 0.f; cur = -1;
  }
  __device__ __forceinline__ void flush(float* __restrict__ acc, int AW, int C, int lane, int priv, bool with_cnt) {
    if (cur < 0) return;
    float* row = acc + (size_t)cur * AW;
    const int ch = (lane * N) >> 5;
    const bool owner = ((lane * N) & 31) == 0;                    // one lane per channel
#pragma unroll
    for (int r = 0; r < R; ++r) {
      const int c = ch + 32 * r;
      if (owner && c < C && run[r] != 0.f) {
        if (priv) row[c] += run[r];
        else atomicAdd(row + c, run[r]);
      }
      run[r] = 0.f;
    }
    if (with_cnt && lane == 0 && cnt != 0.f) {
      if (priv) row[C] += cnt;
      else atomicAdd(row + C, cnt);
    }
    cnt = 0.f; cur = -1;
  }
  // adds the lanes' values `val[c]` (only lanes with `in`) of label L; all 32 lanes call
  __device__ __forceinline__ void add(const float (&val)[CP], bool in, int L, float n_in, float* __restrict__ acc, int AW, int C, int lane,
                                      int priv, bool with_cnt) {
    if (L != cur) { flush(acc, AW, C, lane, priv, with_cnt); cur = L; }
#pragma unroll
    for (int r = 0; r < R; ++r) {
      float v[N];
#pragma unroll
      for (int i = 0; i < N; ++i) v[i] = (in && i + 32 * r < CP) ? val[(i + 32 * r < CP) ? i + 32 * r : 0] : 0.f;
      warp_reduce_channels<N>(v, lane);
      run[r] += v[0];
    }
    cnt += n_in;
  }
};

// sum of p[g * stride], g = 0..G-1, added in index order (deterministic) with the loads of a batch of 8 in flight together
__device__ __forceinline__ float fold_partials(const float* __restrict__ p, size_t stride, int G) {
  float v = 0.f;
  int g = 0;
  for (; g + 8 <= G; g += 8) {
    float t[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) t[j] = __ldcg(p + (size_t)(g + j) * stride);
#pragma unroll
    for (int j = 0; j < 8; ++j) v += t[j];
  }
  for (; g < G; ++g) v += __ldcg(p + (size_t)g * stride);
  return v;
}

template <int CP>
__global__ void __launch_bounds__(kThreads, 2) disc_fwd_lab_kernel(const LabParams lp) {
  extern __shared__ float smem[];   // means [K][CP+1] | accumulators [priv ? kWarps : 1][K][C+1]
  const FwdParams& prm = lp.f;
  if (prm.target_kind != TGT_LABEL_U8 && __ldcg(prm.ws.not_onehot) != 0) return;   // soft masks: disc_fwd_kernel does the work
  const unsigned char* __restrict__ labels_all = (prm.target_kind == TGT_LABEL_U8) ? (const unsigned char*)prm.target : prm.ws.labels;
  const int C = prm.C, K = prm.K, P = prm.H * prm.W;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int MS = CP + 1, AW = C + 1;
  float* __restrict__ s_mu = smem;
  float* __restrict__ s_acc = smem + K * MS;
  float* __restrict__ my_acc = s_acc + (lp.priv ? warp * K * AW : 0);
  const int n_acc = (lp.priv ? kWarps : 1) * K * AW;
  __shared__ double s_dbl[kWarps][3];
  __shared__ int s_last;
  const int b = blockIdx.x / lp.G, g = blockIdx.x % lp.G;
  const int nb = min(max(__ldg(prm.n_objects + b), 0), K);
  const float* __restrict__ emb = prm.emb + (size_t)b * C * P;
  const unsigned char* __restrict__ lab = labels_all + (size_t)b * P;
  // pixels are dealt to the image's CTAs in interleaved 256-pixel blocks: every CTA sees the same foreground / background
  // mix (contiguous chunks left the CTAs of the background rows idle at the grid barrier)
  const int p_lo = g * kWarps * 32, p_hi = P, p_step = lp.G * kWarps * 32;
  float* __restrict__ part = prm.ws.part + (size_t)blockIdx.x * K * AW;
  double* __restrict__ partq = prm.ws.partq + (size_t)blockIdx.x * 3;

  for (int i = threadIdx.x; i < n_acc; i += kThreads) s_acc[i] = 0.f;
  __syncthreads();

  // ------------------------------------------------------------ phase 1: per-instance sums, counts, q-regulariser
  double q_acc = 0.0, nfg_acc = 0.0;
  WarpRun<CP> wr;
  wr.init();
  for (int p0 = p_lo + warp * 32; p0 < p_hi; p0 += p_step) {
    const int p = p0 + lane;
    const bool live = p < p_hi;
    const int l = live ? (int)__ldg(lab + p) : 255;
    float x[CP];
#pragma unroll
    for (int c = 0; c < CP; ++c) x[c] = (c < C && live) ? __ldg(emb + (size_t)c * P + p) : 0.f;
    if (live) {
      // q-regulariser: (|x * fg|_2 - 1)^2 for EVERY pixel (background adds 1); fg = 1 for any label below K
      const float fg = (l < K) ? 1.f : 0.f;
      float ss = 0.f;
#pragma unroll
      for (int c = 0; c < CP; ++c) { const float tq = x[c] * fg; ss = fmaf(tq, tq, ss); }
      const float l2 = sqrtf(ss);
      q_acc += (double)((l2 - 1.f) * (l2 - 1.f));
      nfg_acc += (double)fg;
    }
    const bool valid = l < nb;
    unsigned rem = __ballot_sync(0xffffffffu, valid);
    while (rem) {
      const int leader = __ffs(rem) - 1;
      const int L = __shfl_sync(0xffffffffu, l, leader);
      const bool in = valid && l == L;
      const unsigned grp = __ballot_sync(0xffffffffu, in);
      wr.add(x, in, L, (float)__popc(grp), my_acc, AW, C, lane, lp.priv, true);
      rem &= ~grp;
    }
  }
  wr.flush(my_acc, AW, C, lane, lp.priv, true);
  q_acc = warp_sum_d(q_acc);
  nfg_acc = warp_sum_d(nfg_acc);
  if (lane == 0) { s_dbl[warp][0] = q_acc; s_dbl[warp][1] = nfg_acc; }
  __syncthreads();
  for (int i = threadIdx.x; i < K * AW; i += kThreads) {
    float v = s_acc[i];
    if (lp.priv)
      for (int w = 1; w < kWarps; ++w) v += s_acc[w * K * AW + i];     // fixed order
    part[i] = v;
  }
  if (threadIdx.x == 0) {
    double q = 0.0, nf = 0.0;
    for (int w = 0; w < kWarps; ++w) { q += s_dbl[w][0]; nf += s_dbl[w][1]; }
    partq[0] = q; partq[1] = nf;
  }
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) s_last = (atomicAdd(prm.ws.tick1 + b, 1u) == (unsigned)lp.G - 1u);
  __syncthreads();
  if (s_last) {
    // ---- the image's last CTA: fold the partials in CTA order, then means / norms / N_b / distance / regulariser
    __threadfence();
    float* __restrict__ sums = prm.ws.sums + (size_t)b * K * AW;
    const float* __restrict__ p0 = prm.ws.part + (size_t)b * lp.G * K * AW;
    for (int i = threadIdx.x; i < K * AW; i += kThreads) sums[i] = fold_partials(p0 + i, (size_t)K * AW, lp.G);
    if (threadIdx.x == 0) {
      double q = 0.0, nf = 0.0;
      for (int gg = 0; gg < lp.G; ++gg) { q += __ldcg(prm.ws.partq + ((size_t)b * lp.G + gg) * 3); nf += __ldcg(prm.ws.partq + ((size_t)b * lp.G + gg) * 3 + 1); }
      prm.ws.qb[2 * b] = q; prm.ws.qb[2 * b + 1] = nf;
    }
    __syncthreads();
    for (int k = warp; k < K; k += kWarps) {
      float v = 0.f, v2 = 0.f, cntk = 0.f;
      if (k < nb) {
        cntk = sums[(size_t)k * AW + C];
        if (lane < C) v = sums[(size_t)k * AW + lane] / cntk;
        if (CP > 32 && lane + 32 < C) v2 = sums[(size_t)k * AW + lane + 32] / cntk;
      }
      float r = 1.f;
      if (k < nb) {
        r = sqrtf(warp_sum(v * v + v2 * v2));
        if (prm.normalize_means) { v = v / r; v2 = v2 / r; }
      }
      if (lane < CP) s_mu[k * MS + lane] = v;
      if (CP > 32 && lane + 32 < CP) s_mu[k * MS + lane + 32] = v2;
      if (lane < C) prm.out_means[((size_t)b * K + k) * C + lane] = v;
      if (CP > 32 && lane + 32 < C) prm.out_means[((size_t)b * K + k) * C + lane + 32] = v2;
      if (lane == 0) prm.ws.rnorm[(size_t)b * K + k] = r;
    }
    __syncthreads();
    float nsum = 0.f, dsum = 0.f, rsum = 0.f;
    for (int k = threadIdx.x; k < nb; k += kThreads) {
      const float ck = sums[(size_t)k * AW + C];
      nsum += (ck == 0.f) ? nanf("") : ck;      // an instance id below n_objects without pixels: NaN like the reference
    }
    if (prm.w_dist != 0.f && nb > 1) {
      for (int ij = threadIdx.x; ij < nb * nb; ij += kThreads) {
        const int i = ij / nb, j = ij % nb;
        if (i == j) continue;
        float e = 0.f;
        for (int c = 0; c < C; ++c) {
          const float t = s_mu[i * MS + c] - s_mu[j * MS + c];
          e = (prm.norm == 2) ? fmaf(t, t, e) : e + fabsf(t);
        }
        if (prm.norm == 2) e = sqrtf(e);
        const float m = fmaxf(2.f * prm.delta_d - e, 0.f);
        dsum = fmaf(m, m, dsum);
      }
    }
    if (prm.w_reg != 0.f) {
      for (int k = threadIdx.x; k < nb; k += kThreads) {
        float e = 0.f;
        for (int c = 0; c < C; ++c) {
          const float t = s_mu[k * MS + c];
          e = (prm.norm == 2) ? fmaf(t, t, e) : e + fabsf(t);
        }
        rsum += (prm.norm == 2) ? sqrtf(e) : e;
      }
    }
    nsum = warp_sum(nsum); dsum = warp_sum(dsum); rsum = warp_sum(rsum);
    __shared__ float s3[3][kWarps];
    if (lane == 0) { s3[0][warp] = nsum; s3[1][warp] = dsum; s3[2][warp] = rsum; }
    __syncthreads();
    if (threadIdx.x == 0) {
      float a = 0.f, d = 0.f, r = 0.f;
      for (int w = 0; w < kWarps; ++w) { a += s3[0][w]; d += s3[1][w]; r += s3[2][w]; }
      prm.ws.Nb[b] = a;
      prm.ws.dist_b[b] = (nb > 1) ? d / (float)(nb * (nb - 1)) : 0.f;
      prm.ws.reg_b[b] = r / (float)nb;
    }
  }

  // ------------------------------------------------------------ the one grid barrier: every image's means are published
  group_barrier(prm.ws.lab_bar, gridDim.x);

  for (int i = threadIdx.x; i < K * CP; i += kThreads) {
    const int k = i / CP, c = i % CP;
    s_mu[k * MS + c] = (c < C) ? __ldcg(prm.out_means + ((size_t)b * K + k) * C + c) : 0.f;
  }
  for (int i = threadIdx.x; i < n_acc; i += kThreads) s_acc[i] = 0.f;
  __syncthreads();

  // ------------------------------------------------------------ phase 2: hinge sum + per-instance hinge-gradient sums
  double var_acc = 0.0;
  wr.init();
  for (int p0 = p_lo + warp * 32; p0 < p_hi; p0 += p_step) {
    const int p = p0 + lane;
    const bool live = p < p_hi;
    const int l = live ? (int)__ldg(lab + p) : 255;
    const bool valid = l < nb;
    if (!__any_sync(0xffffffffu, valid)) continue;
    float x[CP];
#pragma unroll
    for (int c = 0; c < CP; ++c) x[c] = (c < C && valid) ? __ldg(emb + (size_t)c * P + p) : 0.f;
    float dir[CP];
#pragma unroll
    for (int c = 0; c < CP; ++c) dir[c] = 0.f;
    float gs = 0.f;
    if (valid) var_acc += (double)hinge_pair<CP>(x, s_mu + l * MS, C, prm.norm, prm.delta_v, 1.f, dir, gs);
#pragma unroll
    for (int c = 0; c < CP; ++c) dir[c] *= gs;
    unsigned rem = __ballot_sync(0xffffffffu, valid);
    while (rem) {
      const int leader = __ffs(rem) - 1;
      const int L = __shfl_sync(0xffffffffu, l, leader);
      const bool in = valid && l == L;
      const unsigned grp = __ballot_sync(0xffffffffu, in);
      wr.add(dir, in, L, 0.f, my_acc, AW, C, lane, lp.priv, false);
      rem &= ~grp;
    }
  }
  wr.flush(my_acc, AW, C, lane, lp.priv, false);
  var_acc = warp_sum_d(var_acc);
  if (lane == 0) s_dbl[warp][2] = var_acc;
  __syncthreads();
  for (int i = threadIdx.x; i < K * AW; i += kThreads) {
    float v = s_acc[i];
    if (lp.priv)
      for (int w = 1; w < kWarps; ++w) v += s_acc[w * K * AW + i];
    part[i] = v;
  }
  if (threadIdx.x == 0) {
    double v = 0.0;
    for (int w = 0; w < kWarps; ++w) v += s_dbl[w][2];
    partq[2] = v;
  }
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) s_last = (atomicAdd(prm.ws.tick2 + b, 1u) == (unsigned)lp.G - 1u);
  __syncthreads();
  if (s_last) {
    __threadfence();
    float* __restrict__ gsum = prm.ws.gsum + (size_t)b * K * C;
    const float* __restrict__ p0 = prm.ws.part + (size_t)b * lp.G * K * AW;
    for (int i = threadIdx.x; i < K * C; i += kThreads) {
      const int k = i / C, c = i % C;
      gsum[i] = fold_partials(p0 + k * AW + c, (size_t)K * AW, lp.G);
    }
    if (threadIdx.x == 0) {
      double v = 0.0;
      for (int gg = 0; gg < lp.G; ++gg) v += __ldcg(prm.ws.partq + ((size_t)b * lp.G + gg) * 3 + 2);
      prm.ws.var_sum[b] = (float)v;
    }
    __threadfence();
    __syncthreads();
    // ---- the last image to finish combines the scalars, images in index order
    if (threadIdx.x == 0) s_last = (atomicAdd(prm.ws.done_cnt, 1u) == (unsigned)prm.bs - 1u);
    __syncthreads();
    if (s_last && threadIdx.x == 0) {
      __threadfence();
      float v = 0.f, d = 0.f, r = 0.f;
      double qs = 0.0, nf = 0.0;
      for (int bb = 0; bb < prm.bs; ++bb) {
        v += __ldcg(prm.ws.var_sum + bb) / __ldcg(prm.ws.Nb + bb);
        d += __ldcg(prm.ws.dist_b + bb);
        r += __ldcg(prm.ws.reg_b + bb);
        qs += __ldcg(prm.ws.qb + 2 * bb);
        nf += __ldcg(prm.ws.qb + 2 * bb + 1);
      }
      *prm.ws.qsum = qs;
      *prm.ws.nfg = nf;                 // the backward reads the foreground count from here
      const float inv_bs = 1.f / (float)prm.bs;
      // discriminative.py:153-159: num = int(sum(target)); loss = sum(...)/num
      const double qden = prm.q_den ? (double)__ldg(prm.q_den) : (double)(long long)nf;
      const float qreg = (float)(qs / qden);
      const float var_t = v * inv_bs;
      const float dist_t = (prm.w_dist != 0.f) ? d * inv_bs : 0.f;
      const float reg_t = (prm.w_reg != 0.f) ? r * inv_bs : 0.f;
      prm.out_terms[0] = var_t; prm.out_terms[1] = dist_t; prm.out_terms[2] = reg_t; prm.out_terms[3] = qreg;
      float loss = 0.f;
      if (prm.w_var != 0.f) loss += prm.w_var * var_t;
      if (prm.w_dist != 0.f) loss += prm.w_dist * dist_t;
      if (prm.w_reg != 0.f) loss += prm.w_reg * reg_t;
      if (prm.w_q != 0.f) loss += prm.w_q * qreg;
      prm.out_loss[0] = loss;
    }
  }
}

// ---------------------------------------------------------------- backward
struct BwdParams {
  const float* emb;
  const void* target;
  const int* n_objects;
  int target_kind;
  int bs, C, H, W, K;
  float delta_v, delta_d;
  int norm;
  int normalize_means;
  float w_var, w_dist, w_reg, w_q;
  DiscWs ws;
  const float* means;       // [bs][K][C] forward output
  const float* grad_loss;   // [1] device scalar
  const float* grad_means;  // [bs][K][C] or null
  const float* q_den;       // see FwdParams
  float* grad_emb;          // [bs][C][P]
};

// One CTA per image: T_k = dL/d(mu~_k) / count_k  for k < n_b.
__global__ void __launch_bounds__(128) disc_bwd_prep_kernel(const BwdParams prm) {
  extern __shared__ float sm[];  // Gam [K][C]
  const int b = blockIdx.x, C = prm.C, K = prm.K;
  const int nb = min(max(__ldg(prm.n_objects + b), 0), K);
  const float go = __ldg(prm.grad_loss);
  const float inv_bs = 1.f / (float)prm.bs;
  const float Nb = prm.ws.Nb[b];
  const float cdir = go * prm.w_var * inv_bs / Nb;
  const float* mu = prm.means + (size_t)b * K * C;
  const float* gsum = prm.ws.gsum + (size_t)b * K * C;
  // Gamma_k = dL/dmu_k
  for (int i = threadIdx.x; i < nb * C; i += blockDim.x) {
    const int k = i / C, c = i % C;
    float gam = -cdir * gsum[i];
    if (prm.grad_means) gam += prm.grad_means[((size_t)b * K + k) * C + c];
    if (prm.w_reg != 0.f) {
      const float cr = go * prm.w_reg * inv_bs / (float)nb;
      if (prm.norm == 2) {
        float e = 0.f;
        for (int cc = 0; cc < C; ++cc) e = fmaf(mu[k * C + cc], mu[k * C + cc], e);
        e = sqrtf(e);
        if (e > 0.f) gam += cr * mu[k * C + c] / e;
      } else {
        const float t = mu[k * C + c];
        gam += cr * ((t > 0.f) ? 1.f : ((t < 0.f) ? -1.f : 0.f));
      }
    }
    if (prm.w_dist != 0.f && nb > 1) {
      const float cd = go * prm.w_dist * inv_bs / (float)(nb * (nb - 1));
      float acc = 0.f;
      for (int j = 0; j < nb; ++j) {
        if (j == k) continue;
        float e = 0.f;
        for (int cc = 0; cc < C; ++cc) {
          const float t = mu[k * C + cc] - mu[j * C + cc];
          e = (prm.norm == 2) ? fmaf(t, t, e) : e + fabsf(t);
        }
        if (prm.norm == 2) e = sqrtf(e);
        const float m = fmaxf(2.f * prm.delta_d - e, 0.f);
        if (m > 0.f) {
          const float t = mu[k * C + c] - mu[j * C + c];
          if (prm.norm == 2) { if (e > 0.f) acc -= 4.f * m * t / e; }
          else acc -= 4.f * m * ((t > 0.f) ? 1.f : ((t < 0.f) ? -1.f : 0.f));
        }
      }
      gam += cd * acc;
    }
    sm[i] = gam;
  }
  __syncthreads();
  for (int i = threadIdx.x; i < K * C; i += blockDim.x) {
    const int k = i / C, c = i % C;
    float t = 0.f;
    if (k < nb) {
      const float cntk = prm.ws.sums[((size_t)b * K + k) * (C + 1) + C];
      float gam = sm[i];
      if (prm.normalize_means) {
        float dot = 0.f;
        for (int cc = 0; cc < C; ++cc) dot = fmaf(mu[k * C + cc], sm[k * C + cc], dot);
        gam = (gam - mu[k * C + c] * dot) / prm.ws.rnorm[(size_t)b * K + k];
      }
      t = gam / cntk;
    }
    prm.ws.T[(size_t)b * K * C + i] = t;
  }
  if (threadIdx.x == 0) {
    prm.ws.coef[b] = cdir;
    if (b == 0) {
      const double nf = *prm.ws.nfg;
      const double qden = prm.q_den ? (double)__ldg(prm.q_den) : (double)(long long)nf;
      prm.ws.coef[prm.bs] = (float)((double)(go * prm.w_q) / qden);
    }
  }
}

template <int CP, int KIND>
__device__ __forceinline__ void disc_bwd_body(const BwdParams& prm, const void* __restrict__ target) {
  extern __shared__ float sm[];  // mu [K][CP+1], T [K][CP+1]
  const int C = prm.C, K = prm.K, P = prm.H * prm.W;
  const int MS = CP + 1;
  const int b = blockIdx.y;
  const int nb = min(max(__ldg(prm.n_objects + b), 0), K);
  float* s_mu = sm;
  float* s_T = sm + K * MS;
  for (int i = threadIdx.x; i < K * C; i += kThreads) {
    const int k = i / C, c = i % C;
    s_mu[k * MS + c] = prm.means[(size_t)b * K * C + i];
    s_T[k * MS + c] = prm.ws.T[(size_t)b * K * C + i];
  }
  __syncthreads();
  const float cdir = prm.ws.coef[b];
  const float cq = prm.ws.coef[prm.bs];
  const float* __restrict__ emb = prm.emb + (size_t)b * C * P;
  float* __restrict__ gout = prm.grad_emb + (size_t)b * C * P;
  const size_t img_off_px = (size_t)b * P;
  for (int p = blockIdx.x * kThreads + threadIdx.x; p < P; p += gridDim.x * kThreads) {
    int k1; float w1, fg;
    const int nnz = read_mask<KIND>(target, img_off_px, p, P, K, k1, w1, fg);
    float x[CP], gr[CP];
#pragma unroll
    for (int c = 0; c < CP; ++c) x[c] = (c < C) ? __ldg(emb + (size_t)c * P + p) : 0.f;
    // q-regulariser: d/dx (|x fg| - 1)^2 = 2 (l-1) fg^2 x / l
    float ss = 0.f;
#pragma unroll
    for (int c = 0; c < CP; ++c) { const float tq = x[c] * fg; ss = fmaf(tq, tq, ss); }
    const float l2 = sqrtf(ss);
    const float qs = (l2 > 0.f) ? cq * 2.f * (l2 - 1.f) * fg * fg / l2 : 0.f;
#pragma unroll
    for (int c = 0; c < CP; ++c) gr[c] = qs * x[c];
    if (nnz == 1) {
      if (k1 < nb) {
        float dir[CP]; float gs;
        hinge_pair<CP>(x, s_mu + k1 * MS, C, prm.norm, prm.delta_v, w1, dir, gs);
#pragma unroll
        for (int c = 0; c < CP; ++c)
          if (c < C) gr[c] += cdir * gs * dir[c] + w1 * s_T[k1 * MS + c];
      }
    } else if (nnz > 1) {
      for (int k = k1; k < nb; ++k) {
        const float m = read_mask_k<KIND>(target, img_off_px, p, P, K, k);
        if (m != 0.f) {
          float dir[CP]; float gs;
          hinge_pair<CP>(x, s_mu + k * MS, C, prm.norm, prm.delta_v, m, dir, gs);
#pragma unroll
          for (int c = 0; c < CP; ++c)
            if (c < C) gr[c] += cdir * gs * dir[c] + m * s_T[k * MS + c];
        }
      }
    }
#pragma unroll
    for (int c = 0; c < CP; ++c)
      if (c < C) gout[(size_t)c * P + p] = gr[c];
  }
}

template <int CP, int KIND>
__global__ void __launch_bounds__(kThreads) disc_bwd_kernel(const BwdParams prm) {
  if (KIND == TGT_LABEL_U8) {
    disc_bwd_body<CP, TGT_LABEL_U8>(prm, prm.target);
  } else if (__ldcg(prm.ws.not_onehot) == 0) {
    disc_bwd_body<CP, TGT_LABEL_U8>(prm, prm.ws.labels);
  } else {
    disc_bwd_body<CP, KIND>(prm, prm.target);
  }
}

// Dense one-hot mask -> u8 label map (255 = background); *flag |= 1 if some
// pixel is not one-hot (several non-zeros, or a value other than 1).
template <int KIND>
__global__ void onehot_to_labels_kernel(const void* __restrict__ tgt, unsigned char* __restrict__ labels, int bs, int K, int P, int* flag,
                                        unsigned long long* fg_count) {
  const size_t total = (size_t)bs * P;
  unsigned cnt = 0;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const int b = (int)(i / P), p = (int)(i % P);
    int k1; float w1, fg;
    const int nnz = read_mask<KIND>(tgt, (size_t)b * P, p, P, K, k1, w1, fg);
    labels[i] = (nnz >= 1) ? (unsigned char)k1 : (unsigned char)255;
    cnt += (nnz >= 1);
    if (nnz > 1 || (nnz == 1 && w1 != 1.f)) atomicOr(flag, 1);
  }
  if (fg_count) {   // integer atomics: order independent, deterministic
    cnt = __reduce_add_sync(0xffffffffu, cnt);
    if ((threadIdx.x & 31) == 0 && cnt) atomicAdd(fg_count, (unsigned long long)cnt);
  }
}

// foreground pixels (label < K) of a u8 label map
__global__ void label_fg_count_kernel(const unsigned char* __restrict__ labels, size_t total, int K, unsigned long long* fg_count) {
  unsigned cnt = 0;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) cnt += (labels[i] < K);
  cnt = __reduce_add_sync(0xffffffffu, cnt);
  if ((threadIdx.x & 31) == 0 && cnt) atomicAdd(fg_count, (unsigned long long)cnt);
}

int allow_smem(const void* fn, size_t smem) {
  if (smem > 48 * 1024) ISA_CUDA(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  return ISA_OK;
}

template <int CP>
int launch_bwd(const BwdParams& prm, dim3 grid, size_t smem, cudaStream_t stream) {
  if (smem > 48 * 1024) {
    int rc = 0;
    switch (prm.target_kind) {
      case TGT_LABEL_U8: rc = allow_smem((const void*)disc_bwd_kernel<CP, TGT_LABEL_U8>, smem); break;
      case TGT_DENSE_F32: rc = allow_smem((const void*)disc_bwd_kernel<CP, TGT_DENSE_F32>, smem); break;
      case TGT_DENSE_I64: rc = allow_smem((const void*)disc_bwd_kernel<CP, TGT_DENSE_I64>, smem); break;
      default: rc = allow_smem((const void*)disc_bwd_kernel<CP, TGT_DENSE_U8>, smem); break;
    }
    if (rc) return rc;
  }
  switch (prm.target_kind) {
    case TGT_LABEL_U8: disc_bwd_kernel<CP, TGT_LABEL_U8><<<grid, kThreads, smem, stream>>>(prm); break;
    case TGT_DENSE_F32: disc_bwd_kernel<CP, TGT_DENSE_F32><<<grid, kThreads, smem, stream>>>(prm); break;
    case TGT_DENSE_I64: disc_bwd_kernel<CP, TGT_DENSE_I64><<<grid, kThreads, smem, stream>>>(prm); break;
    default: disc_bwd_kernel<CP, TGT_DENSE_U8><<<grid, kThreads, smem, stream>>>(prm); break;
  }
  ISA_CUDA(cudaGetLastError());
  return ISA_OK;
}

int launch_onehot_to_labels(const void* target, int target_kind, int bs, int K, int P, unsigned char* labels, int* flag, int num_sms,
                            cudaStream_t stream, unsigned long long* fg_count = nullptr) {
  const size_t total = (size_t)bs * P;
  int grid = (int)((total + 255) / 256);
  if (grid > num_sms * 16) grid = num_sms * 16;
  if (target_kind == TGT_DENSE_F32) onehot_to_labels_kernel<TGT_DENSE_F32><<<grid, 256, 0, stream>>>(target, labels, bs, K, P, flag, fg_count);
  else if (target_kind == TGT_DENSE_I64) onehot_to_labels_kernel<TGT_DENSE_I64><<<grid, 256, 0, stream>>>(target, labels, bs, K, P, flag, fg_count);
  else onehot_to_labels_kernel<TGT_DENSE_U8><<<grid, 256, 0, stream>>>(target, labels, bs, K, P, flag, fg_count);
  ISA_CUDA(cudaGetLastError());
  return ISA_OK;
}

int pick_cp(int C) { return C <= 8 ? 8 : C <= 16 ? 16 : C <= 24 ? 24 : C <= 32 ? 32 : 64; }

int check_common(int target_kind, int bs, int C, int H, int W, int K, int norm) {
  ISA_CHECK_ARG(target_kind >= 0 && target_kind <= 3, "disc_loss: target_kind %d not in 0..3", target_kind);
  ISA_CHECK_ARG(bs > 0 && C > 0 && H > 0 && W > 0 && K > 0, "disc_loss: non-positive dimension (bs=%d C=%d H=%d W=%d K=%d)", bs, C, H, W, K);
  ISA_CHECK_ARG(C <= 64, "disc_loss: embedding width C=%d > 64 is not supported", C);
  ISA_CHECK_ARG(K <= 254, "disc_loss: K=%d > 254 instances (u8 label map limit)", K);
  ISA_CHECK_ARG((long long)H * W < (1ll << 30), "disc_loss: H*W too large");
  ISA_CHECK_ARG(norm == 1 || norm == 2, "disc_loss: norm must be 1 or 2 (got %d)", norm);
  return ISA_OK;
}

const void* lab_kernel_fn(int CP) {
  switch (CP) {
    case 8: return (const void*)disc_fwd_lab_kernel<8>;
    case 16: return (const void*)disc_fwd_lab_kernel<16>;
    case 24: return (const void*)disc_fwd_lab_kernel<24>;
    case 32: return (const void*)disc_fwd_lab_kernel<32>;
    default: return (const void*)disc_fwd_lab_kernel<64>;
  }
}

template <int CP>
const void* col_kernel_fn_cp(int kind) {
  switch (kind) {
    case TGT_LABEL_U8: return (const void*)disc_fwd_kernel<CP, TGT_LABEL_U8>;
    case TGT_DENSE_F32: return (const void*)disc_fwd_kernel<CP, TGT_DENSE_F32>;
    case TGT_DENSE_I64: return (const void*)disc_fwd_kernel<CP, TGT_DENSE_I64>;
    default: return (const void*)disc_fwd_kernel<CP, TGT_DENSE_U8>;
  }
}
const void* col_kernel_fn(int CP, int kind) {
  switch (CP) {
    case 8: return col_kernel_fn_cp<8>(kind);
    case 16: return col_kernel_fn_cp<16>(kind);
    case 24: return col_kernel_fn_cp<24>(kind);
    case 32: return col_kernel_fn_cp<32>(kind);
    default: return col_kernel_fn_cp<64>(kind);
  }
}

// Whether `fn` can take `smem` bytes of dynamic shared memory on top of its static ones; if so, opts it in.
int smem_fits(const void* fn, size_t smem, const IsaDeviceInfo& di, bool* fits) {
  cudaFuncAttributes fa;
  ISA_CUDA(cudaFuncGetAttributes(&fa, fn));
  *fits = smem + fa.sharedSizeBytes <= (size_t)di.max_smem_optin;
  return *fits ? allow_smem(fn, smem) : ISA_OK;
}

// What isa_disc_loss_fwd / isa_disc_loss_bwd launch (see isa_disc_loss_plan).  Decided on the host from the sizes and
// the device alone, before anything is enqueued, so that a refused call leaves every buffer untouched.
struct DiscPlan {
  int route;                 // ISA_DISC_ROUTE_*; -1 when only the backward was planned
  int CP;
  int priv, lab_G, lab_grid; // label-map kernel
  size_t lab_smem;
  int col_G, col_grid;       // column walk
  int strips, rowsplits, rpt;
  size_t col_smem;
  size_t prep_smem;          // backward: disc_bwd_prep_kernel, then disc_bwd_kernel on a (bwd_gx, bs) grid
  int bwd_gx;
  size_t bwd_smem;
};

int make_plan(int target_kind, int bs, int C, int K, int H, int W, bool fwd, const IsaDeviceInfo& di, DiscPlan* pl) {
  DiscPlan& p = *pl;
  const int P = H * W;
  p = DiscPlan{};
  p.route = -1;
  p.CP = pick_cp(C);
  p.priv = -1;

  // ---- backward: the prep kernel's [K][C] Gamma and the streaming kernel's mu and T in shared memory
  ISA_CHECK_ARG(bs <= 65535, "disc_loss: bs=%d > 65535", bs);
  p.prep_smem = sizeof(float) * (size_t)K * C;
  p.bwd_smem = sizeof(float) * 2 * (size_t)K * (p.CP + 1);
  int gx = (P + kThreads - 1) / kThreads;
  const int per_img = (di.num_sms * 8 + bs - 1) / bs;
  if (gx > per_img) gx = per_img;
  p.bwd_gx = gx < 1 ? 1 : gx;
  bool fits = false;
  int rc = smem_fits((const void*)disc_bwd_prep_kernel, p.prep_smem, di, &fits);
  if (rc) return rc;
  if (!fits) { isa_set_error("disc_loss_bwd: prep kernel needs %zu B of shared memory", p.prep_smem); return ISA_ERR_UNSUPPORTED; }
  if (!fwd) return ISA_OK;

  // ---- label-map forward (one grid barrier, deterministic): label maps, and dense masks that turn out one-hot
  const size_t acc1 = sizeof(float) * (size_t)K * (C + 1), mu = sizeof(float) * (size_t)K * (p.CP + 1);
  const int priv = (mu + kWarps * acc1 <= 100 * 1024) ? 1 : 0;
  const size_t lab_smem = mu + (priv ? kWarps : 1) * acc1;
  const void* lab_fn = lab_kernel_fn(p.CP);
  bool use_lab = false;
  rc = smem_fits(lab_fn, lab_smem, di, &fits);
  if (rc) return rc;
  if (fits) {
    int occ = 0;
    ISA_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, lab_fn, kThreads, lab_smem));
    if (occ > 2) occ = 2;
    int nbc = di.num_sms * occ;
    if (nbc > kLabMaxCtas) nbc = kLabMaxCtas;
    if (occ >= 1 && bs <= nbc) {
      use_lab = true;
      int G = nbc / bs;
      const int maxG = (P + 255) / 256;          // no point in CTAs with fewer than one warp-round of pixels
      if (G > maxG) G = maxG;
      if (G < 1) G = 1;
      p.priv = priv;
      p.lab_G = G;
      p.lab_grid = G * bs;
      p.lab_smem = lab_smem;
    }
  }
  if (use_lab && target_kind == TGT_LABEL_U8) { p.route = ROUTE_LAB; return ISA_OK; }

  // ---- column-walk forward: soft / overlapping dense masks (and the fallback when the label-map kernel does not fit).
  // On a dense target it always runs first: it finds out whether the masks are one-hot.
  const size_t smem = sizeof(float) * ((size_t)K * (p.CP + 1) + (size_t)K * (2 * C + 1) + (size_t)kWarps * 32 * ((C + 1) | 1));
  const void* col_fn = col_kernel_fn(p.CP, target_kind);
  rc = smem_fits(col_fn, smem, di, &fits);
  if (rc) return rc;
  int occ = 0;
  if (fits) ISA_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, col_fn, kThreads, smem));
  if (occ < 1) {
    isa_set_error("disc_loss_fwd: the column-walk kernel needs %zu B of shared memory at C=%d K=%d (more than an SM has); it runs "
                  "for every dense target and for label maps with bs=%d above the co-resident CTAs", smem, C, K, bs);
    return ISA_ERR_UNSUPPORTED;
  }
  const int NB = di.num_sms * occ;  // co-resident CTAs
  int G, grid;
  if (bs <= NB) { G = NB / bs; grid = G * bs; } else { G = 1; grid = NB; }
  p.col_G = G;
  p.col_grid = grid;
  p.col_smem = smem;
  p.strips = (W + 31) / 32;
  int rowsplits = (G * kWarps) / p.strips;
  rowsplits = rowsplits < 1 ? 1 : (rowsplits > H ? H : rowsplits);
  p.rpt = (H + rowsplits - 1) / rowsplits;
  p.rowsplits = (H + p.rpt - 1) / p.rpt;
  p.route = use_lab ? ROUTE_COL_THEN_LAB : ROUTE_COL;
  return ISA_OK;
}

}  // namespace

extern "C" {

size_t isa_disc_loss_workspace_bytes(int bs, int C, int K, int H, int W) {
  if (bs <= 0 || C <= 0 || K <= 0 || H <= 0 || W <= 0) return 0;
  return carve(nullptr, bs, C, K, H * W).total_bytes;
}

int isa_disc_loss_plan(int target_kind, int bs, int C, int K, int H, int W, int* h_plan) {
  int rc = check_common(target_kind, bs, C, H, W, K, 2);
  if (rc) return rc;
  ISA_CHECK_ARG(h_plan, "disc_loss_plan: null pointer");
  IsaDeviceInfo di;
  rc = isa_device_info(&di);
  if (rc) return rc;
  DiscPlan pl;
  rc = make_plan(target_kind, bs, C, K, H, W, true, di, &pl);
  if (rc) return rc;
  const int v[] = {pl.route, pl.CP, pl.priv, pl.lab_G, pl.lab_grid, (int)pl.lab_smem, pl.col_G, pl.col_grid, (int)pl.col_smem,
                   (int)pl.prep_smem, pl.bwd_gx, (int)pl.bwd_smem};
  static_assert(sizeof(v) / sizeof(v[0]) == 12, "ISA_DISC_PLAN_LEN");
  for (int i = 0; i < 12; ++i) h_plan[i] = v[i];
  return ISA_OK;
}

int isa_disc_loss_fwd(const float* emb, const void* target, int target_kind, const int* n_objects,
                      int bs, int C, int H, int W, int K,
                      float delta_v, float delta_d, int norm, int normalize_means,
                      float w_var, float w_dist, float w_reg, float w_q,
                      const float* q_den, float* out_loss, float* out_terms, float* out_means,
                      void* workspace, size_t workspace_bytes, cudaStream_t stream) {
  int rc = check_common(target_kind, bs, C, H, W, K, norm);
  if (rc) return rc;
  ISA_CHECK_ARG(emb && target && n_objects && out_loss && out_terms && out_means && workspace, "disc_loss_fwd: null pointer");
  FwdParams prm;
  prm.ws = carve(workspace, bs, C, K, H * W);
  if (workspace_bytes < prm.ws.total_bytes) {
    isa_set_error("disc_loss_fwd: workspace %zu < required %zu bytes", workspace_bytes, prm.ws.total_bytes);
    return ISA_ERR_WORKSPACE;
  }
  IsaDeviceInfo di;
  rc = isa_device_info(&di);
  if (rc) return rc;
  prm.emb = emb; prm.target = target; prm.n_objects = n_objects; prm.target_kind = target_kind;
  prm.bs = bs; prm.C = C; prm.H = H; prm.W = W; prm.K = K;
  prm.delta_v = delta_v; prm.delta_d = delta_d; prm.norm = norm; prm.normalize_means = normalize_means;
  prm.w_var = w_var; prm.w_dist = w_dist; prm.w_reg = w_reg; prm.w_q = w_q;
  prm.out_loss = out_loss; prm.out_terms = out_terms; prm.out_means = out_means; prm.q_den = q_den;

  DiscPlan pl;
  rc = make_plan(target_kind, bs, C, K, H, W, true, di, &pl);
  if (rc) return rc;

  ISA_CUDA(cudaMemsetAsync(workspace, 0, prm.ws.zero_bytes, stream));
  if (target_kind != TGT_LABEL_U8) {
    rc = launch_onehot_to_labels(target, target_kind, bs, K, H * W, prm.ws.labels, prm.ws.not_onehot, di.num_sms, stream);
    if (rc) return rc;
  }
  if (pl.route != ROUTE_LAB) {
    prm.G = pl.col_G; prm.strips = pl.strips; prm.rowsplits = pl.rowsplits; prm.rpt = pl.rpt;
    prm.lab_kernel_follows = (pl.route == ROUTE_COL_THEN_LAB) ? 1 : 0;
    void* args[] = {(void*)&prm};
    ISA_CUDA(cudaLaunchCooperativeKernel(col_kernel_fn(pl.CP, target_kind), dim3(pl.col_grid), dim3(kThreads), args, pl.col_smem, stream));
  }
  if (pl.route != ROUTE_COL) {
    LabParams lp;
    lp.f = prm;
    lp.f.G = 1; lp.f.strips = 0; lp.f.rowsplits = 0; lp.f.rpt = 0; lp.f.lab_kernel_follows = 0;
    lp.G = pl.lab_G;
    lp.chunk = (((H * W + pl.lab_G - 1) / pl.lab_G) + 31) / 32 * 32;
    lp.priv = pl.priv;
    void* args[] = {(void*)&lp};
    ISA_CUDA(cudaLaunchCooperativeKernel(lab_kernel_fn(pl.CP), dim3(pl.lab_grid), dim3(kThreads), args, pl.lab_smem, stream));
  }
  return ISA_OK;
}

int isa_disc_loss_bwd(const float* emb, const void* target, int target_kind, const int* n_objects,
                      int bs, int C, int H, int W, int K,
                      float delta_v, float delta_d, int norm, int normalize_means,
                      float w_var, float w_dist, float w_reg, float w_q,
                      const float* q_den, const float* means, const float* grad_loss, const float* grad_means,
                      float* grad_emb, void* workspace, size_t workspace_bytes, cudaStream_t stream) {
  int rc = check_common(target_kind, bs, C, H, W, K, norm);
  if (rc) return rc;
  ISA_CHECK_ARG(emb && target && n_objects && means && grad_loss && grad_emb && workspace, "disc_loss_bwd: null pointer");
  BwdParams prm;
  prm.ws = carve(workspace, bs, C, K, H * W);
  if (workspace_bytes < prm.ws.total_bytes) {
    isa_set_error("disc_loss_bwd: workspace %zu < required %zu bytes", workspace_bytes, prm.ws.total_bytes);
    return ISA_ERR_WORKSPACE;
  }
  IsaDeviceInfo di;
  rc = isa_device_info(&di);
  if (rc) return rc;
  prm.emb = emb; prm.target = target; prm.n_objects = n_objects; prm.target_kind = target_kind;
  prm.bs = bs; prm.C = C; prm.H = H; prm.W = W; prm.K = K;
  prm.delta_v = delta_v; prm.delta_d = delta_d; prm.norm = norm; prm.normalize_means = normalize_means;
  prm.w_var = w_var; prm.w_dist = w_dist; prm.w_reg = w_reg; prm.w_q = w_q;
  prm.means = means; prm.grad_loss = grad_loss; prm.grad_means = grad_means; prm.grad_emb = grad_emb; prm.q_den = q_den;

  DiscPlan pl;
  rc = make_plan(target_kind, bs, C, K, H, W, false, di, &pl);
  if (rc) return rc;

  disc_bwd_prep_kernel<<<bs, 128, pl.prep_smem, stream>>>(prm);
  ISA_CUDA(cudaGetLastError());
  const dim3 grid(pl.bwd_gx, bs);
  switch (pl.CP) {
    case 8: return launch_bwd<8>(prm, grid, pl.bwd_smem, stream);
    case 16: return launch_bwd<16>(prm, grid, pl.bwd_smem, stream);
    case 24: return launch_bwd<24>(prm, grid, pl.bwd_smem, stream);
    case 32: return launch_bwd<32>(prm, grid, pl.bwd_smem, stream);
    default: return launch_bwd<64>(prm, grid, pl.bwd_smem, stream);
  }
}

int isa_onehot_to_labels(const void* target, int target_kind, int bs, int K, int H, int W,
                         unsigned char* labels, int* not_onehot_flag, unsigned long long* fg_count, cudaStream_t stream) {
  ISA_CHECK_ARG(target_kind >= 1 && target_kind <= 3, "onehot_to_labels: target_kind %d is not a dense kind (1..3)", target_kind);
  ISA_CHECK_ARG(target && labels && not_onehot_flag, "onehot_to_labels: null pointer");
  ISA_CHECK_ARG(bs > 0 && K > 0 && K <= 254 && H > 0 && W > 0, "onehot_to_labels: bad dimensions");
  IsaDeviceInfo di;
  int rc = isa_device_info(&di);
  if (rc) return rc;
  ISA_CUDA(cudaMemsetAsync(not_onehot_flag, 0, sizeof(int), stream));
  if (fg_count) ISA_CUDA(cudaMemsetAsync(fg_count, 0, sizeof(unsigned long long), stream));
  return launch_onehot_to_labels(target, target_kind, bs, K, H * W, labels, not_onehot_flag, di.num_sms, stream, fg_count);
}

int isa_label_fg_count(const unsigned char* labels, long long total, int K, unsigned long long* fg_count, cudaStream_t stream) {
  ISA_CHECK_ARG(labels && fg_count && total > 0 && K > 0 && K <= 255, "label_fg_count: bad argument");
  IsaDeviceInfo di;
  int rc = isa_device_info(&di);
  if (rc) return rc;
  ISA_CUDA(cudaMemsetAsync(fg_count, 0, sizeof(unsigned long long), stream));
  long long grid = (total + 1023) / 1024;
  if (grid > di.num_sms * 8) grid = di.num_sms * 8;
  label_fg_count_kernel<<<(int)grid, 256, 0, stream>>>(labels, (size_t)total, K, fg_count);
  ISA_CUDA(cudaGetLastError());
  return ISA_OK;
}

}  // extern "C"
