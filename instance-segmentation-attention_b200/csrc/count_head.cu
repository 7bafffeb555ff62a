// Fused tail of the instance-count branch (archs.ReSeg(count_head=True)): conv4's bias + ReLU epilogue, the global
// average pool, the 64 -> 1 linear layer, the sigmoid, the count-regression loss and the rounding to an integer count
// in one forward, and the gradient of all of it in one streaming backward.
//
//   y = relu(x + conv_bias)            in place over x [bs][P][C] (NHWC, the bias-free conv4 output)
//   pooled[b][c] = mean_p y            s[b] = sigmoid(pooled[b] . w + b)
//   n_pred[b] = clamp(rint(s[b] * K), 1, K)                  (round half to even, like torch.round)
//   loss = mean_b (s[b] - n_objects[b] / K)^2
//
// HBM-bound: the forward reads and writes the map once (bs*P*C*4 bytes each way), the backward reads y and writes gx.
// Deterministic: per-CTA partial sums in the workspace, folded in a fixed order; no float atomics.  The forward counts
// the positive y per (b, c); with it the bias gradient sum_{b,p} gx = w_c / P * sum_b dz_b * npos[b][c] needs no
// reduction over the map, and the backward is a pure broadcast write.
#include "isa_common.cuh"

namespace {

constexpr int CH_THREADS = 256;
constexpr int CH_ROWS = 256;     // positions per CTA
constexpr int CH_MAX_C = 256;

// workspace layout
//   part_sum [bs][chunks][C] f64   per-CTA sums of y
//   part_pos [bs][chunks][C] i32   per-CTA counts of y > 0
//   npos     [bs][C]         i32   counts of y > 0 (read by the backward)
struct ChLayout {
  size_t off_sum, off_pos, off_npos, total;
  long long chunks;
};

__host__ __device__ inline size_t ch_align(size_t x) { return (x + 255) / 256 * 256; }

__host__ __device__ inline ChLayout ch_layout(int bs, long long P, int C) {
  ChLayout L;
  L.chunks = (P + CH_ROWS - 1) / CH_ROWS;
  const size_t n = (size_t)bs * (size_t)L.chunks * (size_t)C;
  size_t o = 0;
  L.off_sum = o;  o += ch_align(sizeof(double) * n);
  L.off_pos = o;  o += ch_align(sizeof(int) * n);
  L.off_npos = o; o += ch_align(sizeof(int) * (size_t)bs * C);
  L.total = o;
  return L;
}

// dL/dz_b of loss = mean_b (s_b - t_b)^2 through the sigmoid; shared by both backward paths so that they agree bit for bit
__device__ __forceinline__ float ch_dz(const float* s, const int* n_objects, const float* grad_loss, int b, int bs, int K) {
  const float sb = s[b];
  const float tb = (float)n_objects[b] / (float)K;
  return grad_loss[0] * 2.f * (sb - tb) / (float)bs * sb * (1.f - sb);
}

// grid (chunks, bs): y = relu(x + bias) in place, per-CTA column sums and positive counts
__global__ void __launch_bounds__(CH_THREADS)
count_head_fwd_kernel(float* __restrict__ x, const float* __restrict__ conv_bias, long long P, int C,
                      unsigned char* __restrict__ ws) {
  const int b = blockIdx.y;
  const long long chunk = blockIdx.x;
  const ChLayout L = ch_layout(gridDim.y, P, C);
  const int G = C >> 2;                     // float4 channel groups per position
  const int R = CH_THREADS / G;             // positions in flight per CTA
  const int g = threadIdx.x % G, r = threadIdx.x / G;
  __shared__ float4 sh_sum[CH_THREADS];
  __shared__ int4 sh_cnt[CH_THREADS];
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
  int4 cnt = make_int4(0, 0, 0, 0);
  if (r < R) {
    const float4 bias = reinterpret_cast<const float4*>(conv_bias)[g];
    const long long p0 = chunk * CH_ROWS;
    const long long p1 = min(p0 + CH_ROWS, P);
    float4* xb = reinterpret_cast<float4*>(x + (size_t)b * P * C);
    for (long long p = p0 + r; p < p1; p += R) {
      float4 v = xb[(size_t)p * G + g];
      v.x = fmaxf(v.x + bias.x, 0.f);
      v.y = fmaxf(v.y + bias.y, 0.f);
      v.z = fmaxf(v.z + bias.z, 0.f);
      v.w = fmaxf(v.w + bias.w, 0.f);
      xb[(size_t)p * G + g] = v;
      acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
      cnt.x += v.x > 0.f; cnt.y += v.y > 0.f; cnt.z += v.z > 0.f; cnt.w += v.w > 0.f;
    }
  }
  sh_sum[threadIdx.x] = acc;
  sh_cnt[threadIdx.x] = cnt;
  __syncthreads();
  if (threadIdx.x < G) {
    double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
    int c0 = 0, c1 = 0, c2 = 0, c3 = 0;
    for (int rr = 0; rr < R; ++rr) {        // fixed order
      const float4 a = sh_sum[rr * G + g];
      const int4 k = sh_cnt[rr * G + g];
      s0 += a.x; s1 += a.y; s2 += a.z; s3 += a.w;
      c0 += k.x; c1 += k.y; c2 += k.z; c3 += k.w;
    }
    const size_t o = ((size_t)b * L.chunks + chunk) * C + 4 * g;
    double* ps = reinterpret_cast<double*>(ws + L.off_sum) + o;
    int* pc = reinterpret_cast<int*>(ws + L.off_pos) + o;
    ps[0] = s0; ps[1] = s1; ps[2] = s2; ps[3] = s3;
    pc[0] = c0; pc[1] = c1; pc[2] = c2; pc[3] = c3;
  }
}

// one CTA: fold the partials per image in chunk order -> pooled, npos; the linear layer, sigmoid, count and loss
__global__ void __launch_bounds__(CH_THREADS)
count_head_finish_kernel(const float* __restrict__ w, const float* __restrict__ lin_b, const int* __restrict__ n_objects,
                         int bs, long long P, int C, int K, float* __restrict__ pooled, float* __restrict__ s,
                         int* __restrict__ n_pred, float* __restrict__ loss, unsigned char* __restrict__ ws) {
  const ChLayout L = ch_layout(bs, P, C);
  const double* ps = reinterpret_cast<const double*>(ws + L.off_sum);
  const int* pc = reinterpret_cast<const int*>(ws + L.off_pos);
  int* npos = reinterpret_cast<int*>(ws + L.off_npos);
  __shared__ double sh[CH_THREADS / 32];
  const int c = threadIdx.x, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  double loss_acc = 0.0;
  for (int b = 0; b < bs; ++b) {
    double prod = 0.0;
    if (c < C) {
      double a = 0.0;
      int k = 0;
      for (long long ch = 0; ch < L.chunks; ++ch) {
        a += ps[((size_t)b * L.chunks + ch) * C + c];
        k += pc[((size_t)b * L.chunks + ch) * C + c];
      }
      const float pf = (float)(a / (double)P);
      pooled[(size_t)b * C + c] = pf;
      npos[(size_t)b * C + c] = k;
      prod = (double)pf * (double)w[c];
    }
    prod = warp_sum_d(prod);
    if (lane == 0) sh[warp] = prod;
    __syncthreads();
    if (threadIdx.x == 0) {
      double z = (double)lin_b[0];
      for (int i = 0; i < CH_THREADS / 32; ++i) z += sh[i];
      const float sf = (float)(1.0 / (1.0 + exp(-z)));
      s[b] = sf;
      const float r = rintf(__fmul_rn(sf, (float)K));
      n_pred[b] = (int)fminf(fmaxf(r, 1.f), (float)K);
      if (loss) {
        const double d = (double)sf - (double)n_objects[b] / (double)K;
        loss_acc += d * d;
      }
    }
    __syncthreads();
  }
  if (threadIdx.x == 0 && loss) loss[0] = (float)(loss_acc / (double)bs);
}

// grid (chunks + 1, bs): gx = (y > 0) dz_b w_c / P over the map; the extra column's first CTA writes the parameter
// gradients from pooled and the positive counts
__global__ void __launch_bounds__(CH_THREADS)
count_head_bwd_kernel(const float* __restrict__ y, const float* __restrict__ pooled, const float* __restrict__ s,
                      const float* __restrict__ w, const int* __restrict__ n_objects, const float* __restrict__ grad_loss,
                      long long P, int C, int K, float* __restrict__ gx, float* __restrict__ dconv_bias,
                      float* __restrict__ dw, float* __restrict__ db, const unsigned char* __restrict__ ws) {
  const int b = blockIdx.y, bs = gridDim.y;
  const ChLayout L = ch_layout(bs, P, C);
  if ((long long)blockIdx.x == L.chunks) {
    if (b != 0) return;
    const int* npos = reinterpret_cast<const int*>(ws + L.off_npos);
    const int c = threadIdx.x;
    if (c < C) {
      double a = 0.0, d = 0.0;
      for (int bb = 0; bb < bs; ++bb) {
        const double dz = (double)ch_dz(s, n_objects, grad_loss, bb, bs, K);
        a += dz * (double)npos[(size_t)bb * C + c];
        d += dz * (double)pooled[(size_t)bb * C + c];
      }
      dconv_bias[c] = (float)(a * (double)w[c] / (double)P);
      dw[c] = (float)d;
    }
    if (c == 0) {
      double a = 0.0;
      for (int bb = 0; bb < bs; ++bb) a += (double)ch_dz(s, n_objects, grad_loss, bb, bs, K);
      db[0] = (float)a;
    }
    return;
  }
  const int G = C >> 2;
  const int R = CH_THREADS / G;
  const int g = threadIdx.x % G, r = threadIdx.x / G;
  if (r >= R) return;
  const float scale = ch_dz(s, n_objects, grad_loss, b, bs, K) / (float)P;
  const float4 w4 = reinterpret_cast<const float4*>(w)[g];
  const float4 coef = make_float4(scale * w4.x, scale * w4.y, scale * w4.z, scale * w4.w);
  const long long p0 = (long long)blockIdx.x * CH_ROWS;
  const long long p1 = min(p0 + CH_ROWS, P);
  const float4* yb = reinterpret_cast<const float4*>(y + (size_t)b * P * C);
  float4* gb = reinterpret_cast<float4*>(gx + (size_t)b * P * C);
  for (long long p = p0 + r; p < p1; p += R) {
    const float4 v = __ldg(yb + (size_t)p * G + g);
    float4 o;
    o.x = v.x > 0.f ? coef.x : 0.f;
    o.y = v.y > 0.f ? coef.y : 0.f;
    o.z = v.z > 0.f ? coef.z : 0.f;
    o.w = v.w > 0.f ? coef.w : 0.f;
    gb[(size_t)p * G + g] = o;
  }
}

bool aligned16(const void* p) { return ((uintptr_t)p & 15) == 0; }

int check_shape(const char* fn, int bs, long long P, int C, int K) {
  ISA_CHECK_ARG(bs >= 1 && bs <= 65535 && P >= 1 && C >= 4 && C <= CH_MAX_C && C % 4 == 0 && K >= 1 && K <= 254,
                "%s: bs=%d P=%lld C=%d K=%d (1 <= bs <= 65535, 1 <= P, C %% 4 == 0 and 4 <= C <= %d, 1 <= K <= 254)", fn,
                bs, P, C, K, CH_MAX_C);
  ISA_CHECK_ARG((P + CH_ROWS - 1) / CH_ROWS < 0x7fffffffLL, "%s: P=%lld too large", fn, P);
  return ISA_OK;
}

}  // namespace

extern "C" size_t isa_count_head_workspace_bytes(int bs, long long P, int C) {
  if (bs < 1 || P < 1 || C < 1) return 0;
  return ch_layout(bs, P, C).total;
}

extern "C" int isa_count_head_fwd(float* x, const float* conv_bias, const float* w, const float* b, const int* n_objects,
                                  int bs, long long P, int C, int K, float* pooled, float* s, int* n_pred, float* loss,
                                  void* workspace, size_t workspace_bytes, void* stream) {
  ISA_CHECK_ARG(x && conv_bias && w && b && pooled && s && n_pred && workspace, "isa_count_head_fwd: null pointer");
  ISA_CHECK_ARG(!loss || n_objects, "isa_count_head_fwd: loss needs n_objects");
  const int rc = check_shape("isa_count_head_fwd", bs, P, C, K);
  if (rc != ISA_OK) return rc;
  ISA_CHECK_ARG(aligned16(x) && aligned16(conv_bias), "isa_count_head_fwd: x and conv_bias must be 16-byte aligned");
  const ChLayout L = ch_layout(bs, P, C);
  if (workspace_bytes < L.total) {
    isa_set_error("isa_count_head_fwd: workspace %zu < %zu", workspace_bytes, L.total);
    return ISA_ERR_WORKSPACE;
  }
  cudaStream_t st = (cudaStream_t)stream;
  count_head_fwd_kernel<<<dim3((unsigned)L.chunks, bs), CH_THREADS, 0, st>>>(x, conv_bias, P, C, (unsigned char*)workspace);
  ISA_CUDA(cudaGetLastError());
  count_head_finish_kernel<<<1, CH_THREADS, 0, st>>>(w, b, n_objects, bs, P, C, K, pooled, s, n_pred, loss,
                                                     (unsigned char*)workspace);
  ISA_CUDA(cudaGetLastError());
  return ISA_OK;
}

extern "C" int isa_count_head_bwd(const float* y, const float* pooled, const float* s, const float* w, const int* n_objects,
                                  const float* grad_loss, int bs, long long P, int C, int K, float* gx, float* dconv_bias,
                                  float* dw, float* db, void* workspace, size_t workspace_bytes, void* stream) {
  ISA_CHECK_ARG(y && pooled && s && w && n_objects && grad_loss && gx && dconv_bias && dw && db && workspace,
                "isa_count_head_bwd: null pointer");
  const int rc = check_shape("isa_count_head_bwd", bs, P, C, K);
  if (rc != ISA_OK) return rc;
  ISA_CHECK_ARG(aligned16(y) && aligned16(gx) && aligned16(w), "isa_count_head_bwd: y, gx and w must be 16-byte aligned");
  const ChLayout L = ch_layout(bs, P, C);
  if (workspace_bytes < L.total) {
    isa_set_error("isa_count_head_bwd: workspace %zu < %zu", workspace_bytes, L.total);
    return ISA_ERR_WORKSPACE;
  }
  count_head_bwd_kernel<<<dim3((unsigned)L.chunks + 1, bs), CH_THREADS, 0, (cudaStream_t)stream>>>(
      y, pooled, s, w, n_objects, grad_loss, P, C, K, gx, dconv_bias, dw, db, (const unsigned char*)workspace);
  ISA_CUDA(cudaGetLastError());
  return ISA_OK;
}
