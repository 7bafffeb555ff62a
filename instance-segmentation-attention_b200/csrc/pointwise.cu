// Channels-last epilogues of the embedding path's library convolutions / projections, and the residual + LayerNorm
// of the attention block.  All are single-pass HBM-bound kernels over token-major [rows][C] fp32 matrices (NHWC
// activations are exactly that with rows = N*H*W):
//
//   bias_act      y = act(x + b)  in place after a bias-free cuDNN convolution, and its backward
//                 gx = gy * (y > 0),  db = column sums of gx  -- ONE read of gy / y instead of PyTorch's three kernels
//                 (threshold_backward, a strided add and a 13-launch reduce_kernel chain measured at 2.4 ms of the
//                 20 ms CVPPP training step).  Column sums are deterministic: per-CTA partials, fixed-order final sum.
//   add_layernorm MultiHeadAttention's `layer_norm(fc(out) + residual)`
//                 (/root/reference/code/lib/archs/modules/utils.py:218-219), forward and backward with the
//                 gamma / beta gradients, one row per thread (d_model = 24 floats live in registers).
#include "isa_common.cuh"
#include "isa_ptx.cuh"
#include "isa_tcgen05.cuh"

namespace {

constexpr int kThreads = 256;

// ------------------------------------------------------------------------------------------------ bias + activation
// V = 4: float4 columns (C % 4 == 0), V = 1: scalar columns.  Thread t < A (A = largest multiple of cv <= 256) owns
// column t % cv for the whole kernel and walks rows with a fixed stride, so a CTA's threads always cover a
// contiguous A*4V-byte span.
template <int V>
struct Vec;
template <>
struct Vec<4> { using T = float4; };
template <>
struct Vec<1> { using T = float; };

__device__ __forceinline__ float4 ld4(const float* p) { return *reinterpret_cast<const float4*>(p); }

template <int V, bool RELU>
__global__ void __launch_bounds__(kThreads) bias_act_fwd_kernel(float* __restrict__ x, const float* __restrict__ bias, long long rows, int C) {
  const int cv = C / V;
  const int rpi = kThreads / cv;                       // rows per CTA iteration
  const int t = threadIdx.x;
  if (t >= rpi * cv) return;
  const int c = (t % cv) * V;
  float b[V];
#pragma unroll
  for (int i = 0; i < V; ++i) b[i] = __ldg(bias + c + i);
  const long long step = (long long)gridDim.x * rpi;
  long long r = (long long)blockIdx.x * rpi + t / cv;
  if (V == 4) {
    // four independent rows per iteration: the loads are issued together (in-place update: the compiler may not hoist
    // a load above the previous row's store on its own)
    for (; r + 3 * step < rows; r += 4 * step) {
      float4 v[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) v[j] = ld4(x + (r + j * step) * C + c);
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        v[j].x += b[0]; v[j].y += b[1 % V]; v[j].z += b[2 % V]; v[j].w += b[3 % V];
        if (RELU) { v[j].x = fmaxf(v[j].x, 0.f); v[j].y = fmaxf(v[j].y, 0.f); v[j].z = fmaxf(v[j].z, 0.f); v[j].w = fmaxf(v[j].w, 0.f); }
        *reinterpret_cast<float4*>(x + (r + j * step) * C + c) = v[j];
      }
    }
  }
  for (; r < rows; r += step) {
    float* p = x + r * C + c;
    if (V == 4) {
      float4 v = ld4(p);
      v.x += b[0]; v.y += b[1 % V]; v.z += b[2 % V]; v.w += b[3 % V];
      if (RELU) { v.x = fmaxf(v.x, 0.f); v.y = fmaxf(v.y, 0.f); v.z = fmaxf(v.z, 0.f); v.w = fmaxf(v.w, 0.f); }
      *reinterpret_cast<float4*>(p) = v;
    } else {
      float v = *p + b[0];
      if (RELU) v = fmaxf(v, 0.f);
      *p = v;
    }
  }
}

// gx = RELU ? gy * (y > 0) : gy (not written when gx == nullptr);  partial[blockIdx][C] = this CTA's column sums
template <int V, bool RELU>
__global__ void __launch_bounds__(kThreads) bias_act_bwd_kernel(const float* __restrict__ gy, const float* __restrict__ y, float* __restrict__ gx,
                                                                float* __restrict__ partial, long long rows, int C) {
  __shared__ float s_acc[kThreads * V];
  const int cv = C / V;
  const int rpi = kThreads / cv;
  const int t = threadIdx.x;
  const bool active = t < rpi * cv;
  const int c = (t % cv) * V;
  float acc[V];
#pragma unroll
  for (int i = 0; i < V; ++i) acc[i] = 0.f;
  if (active) {
    const long long step = (long long)gridDim.x * rpi;
    long long r = (long long)blockIdx.x * rpi + t / cv;
    if (V == 4) {
      // two independent rows per iteration (four 16-byte loads in flight per thread)
      for (; r + step < rows; r += 2 * step) {
        float4 g[2], yy[2];
#pragma unroll
        for (int j = 0; j < 2; ++j) {
          const long long o = (r + j * step) * C + c;
          g[j] = ld4(gy + o);
          if (RELU) yy[j] = ld4(y + o);
        }
#pragma unroll
        for (int j = 0; j < 2; ++j) {
          const long long o = (r + j * step) * C + c;
          if (RELU) {
            g[j].x = yy[j].x > 0.f ? g[j].x : 0.f; g[j].y = yy[j].y > 0.f ? g[j].y : 0.f;
            g[j].z = yy[j].z > 0.f ? g[j].z : 0.f; g[j].w = yy[j].w > 0.f ? g[j].w : 0.f;
          }
          if (gx) *reinterpret_cast<float4*>(gx + o) = g[j];
          acc[0] += g[j].x; acc[1 % V] += g[j].y; acc[2 % V] += g[j].z; acc[3 % V] += g[j].w;
        }
      }
    }
    for (; r < rows; r += step) {
      const long long o = r * C + c;
      if (V == 4) {
        float4 g = ld4(gy + o);
        if (RELU) {
          const float4 yy = ld4(y + o);
          g.x = yy.x > 0.f ? g.x : 0.f; g.y = yy.y > 0.f ? g.y : 0.f; g.z = yy.z > 0.f ? g.z : 0.f; g.w = yy.w > 0.f ? g.w : 0.f;
        }
        if (gx) *reinterpret_cast<float4*>(gx + o) = g;
        acc[0] += g.x; acc[1 % V] += g.y; acc[2 % V] += g.z; acc[3 % V] += g.w;
      } else {
        float g = gy[o];
        if (RELU) g = y[o] > 0.f ? g : 0.f;
        if (gx) gx[o] = g;
        acc[0] += g;
      }
    }
  }
#pragma unroll
  for (int i = 0; i < V; ++i) s_acc[t * V + i] = acc[i];
  __syncthreads();
  if (t < cv) {
    float s[V];
#pragma unroll
    for (int i = 0; i < V; ++i) s[i] = 0.f;
    for (int j = 0; j < rpi; ++j)
#pragma unroll
      for (int i = 0; i < V; ++i) s[i] += s_acc[(j * cv + t) * V + i];
#pragma unroll
    for (int i = 0; i < V; ++i) partial[(size_t)blockIdx.x * C + t * V + i] = s[i];
  }
}

// out[c] = sum over `n` partial rows in a fixed order: 8 row groups x 32 columns per CTA, then the groups in order
__global__ void __launch_bounds__(256) column_reduce_kernel(const float* __restrict__ partial, int n, int C, float* __restrict__ out) {
  __shared__ float s_g[8][32];
  const int c = blockIdx.x * 32 + (threadIdx.x & 31), g = threadIdx.x >> 5;
  float s = 0.f;
  if (c < C)
    for (int i = g; i < n; i += 8) s += partial[(size_t)i * C + c];
  s_g[g][threadIdx.x & 31] = s;
  __syncthreads();
  if (g == 0 && c < C) {
    float t = 0.f;
#pragma unroll
    for (int k = 0; k < 8; ++k) t += s_g[k][threadIdx.x & 31];
    out[c] = t;
  }
}

int bias_act_grid(long long rows, int C, int V, int num_sms) {
  const int cv = C / V;
  const int rpi = kThreads / cv;
  long long g = (rows + rpi - 1) / rpi;
  const long long cap = (long long)num_sms * 4;
  return (int)(g < cap ? g : cap);
}

// ------------------------------------------------------------------------------------------------ residual + LayerNorm
template <int C>
__global__ void __launch_bounds__(kThreads) add_ln_fwd_kernel(const float* __restrict__ x, const float* __restrict__ res, const float* __restrict__ gamma,
                                                              const float* __restrict__ beta, long long rows, float eps, float* __restrict__ y,
                                                              float* __restrict__ stats) {
  const long long r = (long long)blockIdx.x * kThreads + threadIdx.x;
  if (r >= rows) return;
  float v[C];
#pragma unroll
  for (int i = 0; i < C; i += 4) {
    float4 a = ld4(x + r * C + i);
    if (res) { const float4 b = ld4(res + r * C + i); a.x += b.x; a.y += b.y; a.z += b.z; a.w += b.w; }
    v[i] = a.x; v[i + 1] = a.y; v[i + 2] = a.z; v[i + 3] = a.w;
  }
  float mean = 0.f;
#pragma unroll
  for (int i = 0; i < C; ++i) mean += v[i];
  mean *= 1.f / C;
  float var = 0.f;
#pragma unroll
  for (int i = 0; i < C; ++i) { const float d = v[i] - mean; var = fmaf(d, d, var); }
  var *= 1.f / C;
  const float rstd = rsqrtf(var + eps);
#pragma unroll
  for (int i = 0; i < C; i += 4) {
    float4 o;
    o.x = (v[i] - mean) * rstd * __ldg(gamma + i) + __ldg(beta + i);
    o.y = (v[i + 1] - mean) * rstd * __ldg(gamma + i + 1) + __ldg(beta + i + 1);
    o.z = (v[i + 2] - mean) * rstd * __ldg(gamma + i + 2) + __ldg(beta + i + 2);
    o.w = (v[i + 3] - mean) * rstd * __ldg(gamma + i + 3) + __ldg(beta + i + 3);
    *reinterpret_cast<float4*>(y + r * C + i) = o;
  }
  stats[2 * r] = mean;
  stats[2 * r + 1] = rstd;
}

// gv = d loss / d (x + res);  partial[blockIdx][2C] = this CTA's (dgamma | dbeta) sums
template <int C>
__global__ void __launch_bounds__(kThreads) add_ln_bwd_kernel(const float* __restrict__ gy, const float* __restrict__ x, const float* __restrict__ res,
                                                              const float* __restrict__ gamma, const float* __restrict__ stats, long long rows,
                                                              float* __restrict__ gv, float* __restrict__ partial) {
  __shared__ float s_part[kThreads / 32][2 * C];
  const long long r = (long long)blockIdx.x * kThreads + threadIdx.x;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float dg[C], db[C];
  if (r < rows) {
    const float mean = stats[2 * r], rstd = stats[2 * r + 1];
    float xh[C], g[C];
#pragma unroll
    for (int i = 0; i < C; i += 4) {
      float4 a = ld4(x + r * C + i);
      if (res) { const float4 b = ld4(res + r * C + i); a.x += b.x; a.y += b.y; a.z += b.z; a.w += b.w; }
      const float4 q = ld4(gy + r * C + i);
      xh[i] = (a.x - mean) * rstd; xh[i + 1] = (a.y - mean) * rstd; xh[i + 2] = (a.z - mean) * rstd; xh[i + 3] = (a.w - mean) * rstd;
      g[i] = q.x; g[i + 1] = q.y; g[i + 2] = q.z; g[i + 3] = q.w;
    }
    float m1 = 0.f, m2 = 0.f;
#pragma unroll
    for (int i = 0; i < C; ++i) {
      dg[i] = g[i] * xh[i];
      db[i] = g[i];
      const float dxh = g[i] * __ldg(gamma + i);
      m1 += dxh;
      m2 = fmaf(dxh, xh[i], m2);
      g[i] = dxh;
    }
    m1 *= 1.f / C;
    m2 *= 1.f / C;
#pragma unroll
    for (int i = 0; i < C; i += 4) {
      float4 o;
      o.x = rstd * (g[i] - m1 - xh[i] * m2);
      o.y = rstd * (g[i + 1] - m1 - xh[i + 1] * m2);
      o.z = rstd * (g[i + 2] - m1 - xh[i + 2] * m2);
      o.w = rstd * (g[i + 3] - m1 - xh[i + 3] * m2);
      *reinterpret_cast<float4*>(gv + r * C + i) = o;
    }
  } else {
#pragma unroll
    for (int i = 0; i < C; ++i) { dg[i] = 0.f; db[i] = 0.f; }
  }
#pragma unroll
  for (int i = 0; i < C; ++i) {
    const float a = warp_sum(dg[i]), b = warp_sum(db[i]);
    if (lane == 0) { s_part[warp][i] = a; s_part[warp][C + i] = b; }
  }
  __syncthreads();
  if (threadIdx.x < 2 * C) {
    float s = 0.f;
#pragma unroll
    for (int w = 0; w < kThreads / 32; ++w) s += s_part[w][threadIdx.x];
    partial[(size_t)blockIdx.x * 2 * C + threadIdx.x] = s;
  }
}

template <int C>
int launch_ln_fwd(const float* x, const float* res, const float* gamma, const float* beta, long long rows, float eps, float* y, float* stats,
                  cudaStream_t stream) {
  add_ln_fwd_kernel<C><<<(unsigned)((rows + kThreads - 1) / kThreads), kThreads, 0, stream>>>(x, res, gamma, beta, rows, eps, y, stats);
  ISA_CUDA(cudaGetLastError());
  return ISA_OK;
}
template <int C>
int launch_ln_bwd(const float* gy, const float* x, const float* res, const float* gamma, const float* stats, long long rows, float* gv, float* dgamma,
                  float* dbeta, float* partial, cudaStream_t stream) {
  const int grid = (int)((rows + kThreads - 1) / kThreads);
  add_ln_bwd_kernel<C><<<grid, kThreads, 0, stream>>>(gy, x, res, gamma, stats, rows, gv, partial);
  ISA_CUDA(cudaGetLastError());
  // (dgamma | dbeta) are contiguous halves of each partial row
  column_reduce_kernel<<<(2 * C + 31) / 32, 256, 0, stream>>>(partial, grid, 2 * C, partial + (size_t)grid * 2 * C);
  ISA_CUDA(cudaGetLastError());
  ISA_CUDA(cudaMemcpyAsync(dgamma, partial + (size_t)grid * 2 * C, C * sizeof(float), cudaMemcpyDeviceToDevice, stream));
  ISA_CUDA(cudaMemcpyAsync(dbeta, partial + (size_t)grid * 2 * C + C, C * sizeof(float), cudaMemcpyDeviceToDevice, stream));
  return ISA_OK;
}

bool ln_width_ok(int C) { return C == 8 || C == 16 || C == 24 || C == 32 || C == 40 || C == 48 || C == 64; }



// ------------------------------------------------------------------------------------------------ 2x2 / stride-2 max pool
// The backbone's nn.MaxPool2d(2, 2) on NHWC activations (/root/reference/code/lib/archs/modules/vgg16.py:82-140 pools
// between the conv stages).  Forward keeps the window position of the maximum (first maximum in row-major window order,
// NaN wins, like PyTorch) as one byte per output element, so the backward is a pure scatter: read gy + index, write
// the four window positions (PyTorch's NHWC backward re-reads the indices as int64 and measured 2.4x the forward).
__global__ void __launch_bounds__(256) maxpool2x2_fwd_kernel(const float* __restrict__ x, float* __restrict__ y, unsigned char* __restrict__ idx,
                                                             long long total4, int Ho, int Wo, int W, int C4, long long in_img) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total4; i += (long long)gridDim.x * blockDim.x) {
    const int c4 = (int)(i % C4);
    long long r = i / C4;
    const int wo = (int)(r % Wo); r /= Wo;
    const int ho = (int)(r % Ho);
    const long long n = r / Ho;
    const long long base = n * in_img + ((long long)(2 * ho) * W + 2 * wo) * (C4 * 4) + c4 * 4;
    const float4 a = ld4(x + base), b = ld4(x + base + C4 * 4);
    const float4 c = ld4(x + base + (long long)W * C4 * 4), d = ld4(x + base + (long long)W * C4 * 4 + C4 * 4);
    float4 m; unsigned int sel = 0;
#define ISA_POOL1(F, SH)                                                         \
    {                                                                            \
      float best = a.F; unsigned int bi = 0;                                     \
      if (b.F > best || b.F != b.F) { best = b.F; bi = 1; }                      \
      if (c.F > best || c.F != c.F) { best = c.F; bi = 2; }                      \
      if (d.F > best || d.F != d.F) { best = d.F; bi = 3; }                      \
      m.F = best; sel |= bi << SH;                                               \
    }
    ISA_POOL1(x, 0) ISA_POOL1(y, 8) ISA_POOL1(z, 16) ISA_POOL1(w, 24)
#undef ISA_POOL1
    *reinterpret_cast<float4*>(y + i * 4) = m;
    if (idx) *reinterpret_cast<unsigned int*>(idx + i * 4) = sel;
  }
}

// `add` (optional): a second gradient of the pooled tensor's INPUT (the skip connection that also consumed it), read with
// its own pixel stride (a channel slice of a wider NHWC gradient, e.g. what torch.cat's backward hands back) and summed in
// the same pass -- autograd would otherwise materialise the scatter, copy the slice and run a separate add.
__global__ void __launch_bounds__(256) maxpool2x2_bwd_kernel(const float* __restrict__ gy, const unsigned char* __restrict__ idx,
                                                             float* __restrict__ gx, long long total4, int Ho, int Wo, int W, int C4,
                                                             long long in_img, const float* __restrict__ add, long long add_px) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total4; i += (long long)gridDim.x * blockDim.x) {
    const int c4 = (int)(i % C4);
    long long r = i / C4;
    const int wo = (int)(r % Wo); r /= Wo;
    const int ho = (int)(r % Ho);
    const long long n = r / Ho;
    const long long base = n * in_img + ((long long)(2 * ho) * W + 2 * wo) * (C4 * 4) + c4 * 4;
    const float4 g = ld4(gy + i * 4);
    const unsigned int sel = *reinterpret_cast<const unsigned int*>(idx + i * 4);
    const unsigned int s0 = sel & 3u, s1 = (sel >> 8) & 3u, s2 = (sel >> 16) & 3u, s3 = (sel >> 24) & 3u;
    const long long pix0 = n * ((long long)2 * Ho * W) + (long long)(2 * ho) * W + 2 * wo;   // H == 2 Ho whenever `add` is given
#pragma unroll
    for (unsigned int q = 0; q < 4; ++q) {
      float4 o;
      o.x = s0 == q ? g.x : 0.f; o.y = s1 == q ? g.y : 0.f; o.z = s2 == q ? g.z : 0.f; o.w = s3 == q ? g.w : 0.f;
      if (add) {
        const float4 a = ld4(add + (pix0 + (long long)(q >> 1) * W + (q & 1)) * add_px + c4 * 4);
        o.x += a.x; o.y += a.y; o.z += a.z; o.w += a.w;
      }
      *reinterpret_cast<float4*>(gx + base + (long long)(q >> 1) * W * C4 * 4 + (q & 1) * C4 * 4) = o;
    }
  }
}


// ------------------------------------------------------------------------------------------------ fused clip + Adadelta
// The training step's `clip_grad_norm_` + `Adadelta.step` (/root/reference/code/lib/model.py:141-160, 271-281;
// settings: OPTIMIZER = 'Adadelta', CLIP_GRAD_NORM = 10) over ONE flat parameter / gradient / state buffer: a
// sum-of-squares pass (per-CTA double partials) and an update pass that first folds the partials in a fixed order
// (every CTA gets the same norm, no host round trip) -- instead of ~45 multi-tensor launches (0.6 ms per step).
__global__ void __launch_bounds__(256) sumsq_partial_kernel(const float* __restrict__ g, long long n, double* __restrict__ partial) {
  __shared__ double s_w[8];
  double acc = 0.0;
  const long long n4 = n >> 2;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (long long)gridDim.x * blockDim.x) {
    const float4 v = ld4(g + i * 4);
    acc += (double)v.x * v.x + (double)v.y * v.y + (double)v.z * v.z + (double)v.w * v.w;
  }
  if (blockIdx.x == 0 && threadIdx.x < (n & 3)) { const float v = g[n4 * 4 + threadIdx.x]; acc += (double)v * v; }
  acc = warp_sum_d(acc);
  if ((threadIdx.x & 31) == 0) s_w[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0.0;
#pragma unroll
    for (int w = 0; w < 8; ++w) t += s_w[w];
    partial[blockIdx.x] = t;
  }
}

struct AdadeltaParams {
  float* param; const float* grad; float* square_avg; float* acc_delta;
  long long n;
  float lr, rho, eps, weight_decay, max_norm;   // max_norm <= 0: no clipping
  const double* partial; int n_partial;
  float* norm_out;                              // total gradient norm before clipping (or null)
};

__device__ __forceinline__ void adadelta1(float& p, float g, float& sq, float& ad, const AdadeltaParams& a, float clip) {
  g = g * clip;
  if (a.weight_decay != 0.f) g = fmaf(a.weight_decay, p, g);
  sq = a.rho * sq + (1.f - a.rho) * g * g;
  const float delta = sqrtf(ad + a.eps) / sqrtf(sq + a.eps) * g;
  ad = a.rho * ad + (1.f - a.rho) * delta * delta;
  p = p - a.lr * delta;
}

__global__ void __launch_bounds__(256) adadelta_step_kernel(const AdadeltaParams a) {
  __shared__ float s_clip;
  if (threadIdx.x == 0) {
    float clip = 1.f;
    if (a.max_norm > 0.f || a.norm_out) {
      double t = 0.0;
      for (int i = 0; i < a.n_partial; ++i) t += a.partial[i];
      const float norm = (float)sqrt(t);
      if (a.norm_out && blockIdx.x == 0) *a.norm_out = norm;
      if (a.max_norm > 0.f) clip = fminf(a.max_norm / (norm + 1e-6f), 1.f);     // torch.nn.utils.clip_grad_norm_
    }
    s_clip = clip;
  }
  __syncthreads();
  const float clip = s_clip;
  const long long n4 = a.n >> 2;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (long long)gridDim.x * blockDim.x) {
    float4 p = ld4(a.param + i * 4), sq = ld4(a.square_avg + i * 4), ad = ld4(a.acc_delta + i * 4);
    const float4 g = ld4(a.grad + i * 4);
    adadelta1(p.x, g.x, sq.x, ad.x, a, clip); adadelta1(p.y, g.y, sq.y, ad.y, a, clip);
    adadelta1(p.z, g.z, sq.z, ad.z, a, clip); adadelta1(p.w, g.w, sq.w, ad.w, a, clip);
    *reinterpret_cast<float4*>(a.param + i * 4) = p;
    *reinterpret_cast<float4*>(a.square_avg + i * 4) = sq;
    *reinterpret_cast<float4*>(a.acc_delta + i * 4) = ad;
  }
  if (blockIdx.x == 0 && threadIdx.x < (a.n & 3)) {
    const long long i = n4 * 4 + threadIdx.x;
    adadelta1(a.param[i], a.grad[i], a.square_avg[i], a.acc_delta[i], a, clip);
  }
}

__device__ __forceinline__ void cp_async8(void* smem_dst, const void* gsrc) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(smem_u32(smem_dst)), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() {
  asm volatile("cp.async.commit_group;\n\tcp.async.wait_group 0;" ::: "memory");
}

// ------------------------------------------------------------------------------------------------ pixel heads
// The semantic / embedding heads are 1x1 convolutions over the concatenation [up-sampled features | skip]
// (/root/reference/code/lib/archs/reseg.py:122-126).  As plain library ops that is a 478 MB concatenation, two cuDNN
// convolutions that each re-read it, two bias kernels and an NHWC -> NCHW copy of the embedding (the loss and the
// clustering kernels want [C][H*W] planes).  Here: ONE pass that reads the two NHWC sources once, never materialises the
// concatenation, and writes both outputs as NCHW planes; backward = one pass producing both NHWC source gradients.
// Exact fp32 (FFMA); the stacked weights sit in shared memory so one LDS feeds several FMAs of two pixels.
constexpr int kHeadThreads = 128;

struct HeadsParams {
  const float* xa; const float* xb;   // NHWC sources [P][Ca], [P][Cb]  (xb may be NULL with Cb = 0)
  int Ca, Cb;
  const float* w;                     // stacked weights [Co][Ca + Cb]
  const float* bias;                  // [Co] or NULL
  float* out0; float* out1;           // NCHW outputs [n][Co0][HW], [n][Co1][HW]  (Co = Co0 + Co1)
  int Co0, Co1;
  long long P; int HW;
};

// One CTA = 128-pixel tiles, one pixel per thread.  The tile's source rows are contiguous in memory, so they are staged
// into shared memory with fully coalesced 8-byte loads (a thread reading its own 200-byte row straight from global
// touches 32 sectors per load instruction: measured 334 us instead of ~100) and read back with an odd row stride
// (conflict-free); the stacked weights are W^T[k][COP] so one broadcast LDS.128 feeds four output channels.
constexpr int kHeadTile = 128;

template <int COP>   // COP = Co rounded up to a multiple of 4
__global__ void __launch_bounds__(kHeadThreads) pixel_heads_fwd_kernel(const HeadsParams p) {
  extern __shared__ __align__(16) float s_buf[];
  const int K = p.Ca + p.Cb, Co = p.Co0 + p.Co1;
  const int KS = K | 1;                          // odd row stride of the staged tile
  float* s_wt = s_buf;                           // W^T: [K][COP]
  float* s_x = s_buf + K * COP;                  // [kHeadTile][KS]
  for (int i = threadIdx.x; i < K * COP; i += blockDim.x) {
    const int k = i / COP, co = i % COP;
    s_wt[i] = co < Co ? __ldg(p.w + (size_t)co * K + k) : 0.f;
  }
  const long long n_tiles = (p.P + kHeadTile - 1) / kHeadTile;
  for (long long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const long long p0 = tile * kHeadTile;
    const int np = (int)((p.P - p0) < kHeadTile ? (p.P - p0) : kHeadTile);
    __syncthreads();
#pragma unroll 1
    for (int src = 0; src < 2; ++src) {
      const float* __restrict__ x = (src == 0 ? p.xa : p.xb);
      const int Cs = src == 0 ? p.Ca : p.Cb, k0 = src == 0 ? 0 : p.Ca;
      const int half = Cs >> 1;
      const float2* __restrict__ x2 = reinterpret_cast<const float2*>(x + p0 * Cs);
#pragma unroll 4
      for (int i = threadIdx.x; i < np * half; i += kHeadThreads) {
        const float2 v = __ldg(x2 + i);
        const int pp = i / half, k = (i - pp * half) * 2;
        s_x[pp * KS + k0 + k] = v.x;
        s_x[pp * KS + k0 + k + 1] = v.y;
      }
    }
    __syncthreads();
    if ((int)threadIdx.x < np) {
      float acc[COP];
#pragma unroll
      for (int c = 0; c < COP; ++c) acc[c] = 0.f;
      const float* __restrict__ xr = s_x + threadIdx.x * KS;
#pragma unroll 2
      for (int k = 0; k < K; ++k) {
        const float xv = xr[k];
#pragma unroll
        for (int c = 0; c < COP; c += 4) {
          const float4 w = *reinterpret_cast<const float4*>(s_wt + (size_t)k * COP + c);
          acc[c] = fmaf(xv, w.x, acc[c]); acc[c + 1] = fmaf(xv, w.y, acc[c + 1]);
          acc[c + 2] = fmaf(xv, w.z, acc[c + 2]); acc[c + 3] = fmaf(xv, w.w, acc[c + 3]);
        }
      }
      const long long pix = p0 + threadIdx.x;
      const long long n = pix / p.HW, hw = pix - n * p.HW;
#pragma unroll
      for (int c = 0; c < COP; ++c) {
        if (c >= Co) break;
        const float v = acc[c] + (p.bias ? __ldg(p.bias + c) : 0.f);
        if (c < p.Co0) p.out0[(n * p.Co0 + c) * p.HW + hw] = v;
        else p.out1[(n * p.Co1 + (c - p.Co0)) * p.HW + hw] = v;
      }
    }
  }
}


// ---- tensor-core pixel heads (Ca + Cb <= 128, Co <= 32): the FFMA kernels above are bound by the delivery of the weight
// operand from shared memory (a broadcast LDS.128 costs four passes for 16 useful bytes).  Here a 128-pixel tile is a
// [128 x K] x [K x 32] product on tcgen05: every thread converts ITS pixel's row (staged in shared memory by coalesced
// loads) to bf16 hi / lo pairs and writes it into tensor memory as the A operand (TMEM lane = pixel); the stacked weights
// are a K-major bf16 hi / lo B operand built once per CTA; a_hi [b_hi ; b_lo] (N = 64) + a_lo b_hi (N = 32) per k-step
// keeps fp32-level accuracy (error ~2^-16).  The epilogue reads the pixel's 2 x 32 accumulator columns and stores NCHW.
constexpr int kHtKP = 128;                       // padded reduction length
constexpr int kHtSbo = (kHtKP / 8) * 128;        // 2048: byte stride between 8-row groups of a K-major [rows][128] operand
constexpr int kHtWPart = 4 * kHtSbo;             // 32 rows: 8192 bytes per part (hi | lo contiguous = one N = 64 operand)

__global__ void __launch_bounds__(kHeadThreads) pixel_heads_fwd_tc_kernel(const HeadsParams p) {
  extern __shared__ __align__(16) unsigned char smem_raw_h[];
  unsigned char* sm = smem_raw_h + ((128u - (smem_u32(smem_raw_h) & 127u)) & 127u);
  const int K = p.Ca + p.Cb, Co = p.Co0 + p.Co1;
  const int KS = K;                        // even row stride: 8-byte cp.async destinations (row reads are 2-way conflicted)
  unsigned char* s_w = sm;                                               // [W_hi ; W_lo] K-major, 2 x 8192 B
  float* s_x = reinterpret_cast<float*>(sm + 2 * kHtWPart);              // [kHeadTile][KS]
  uint64_t* s_bar = reinterpret_cast<uint64_t*>(s_x + kHeadTile * KS + 1);
  s_bar = reinterpret_cast<uint64_t*>((reinterpret_cast<uintptr_t>(s_bar) + 7) & ~uintptr_t(7));
  uint32_t* s_tmem = reinterpret_cast<uint32_t*>(s_bar + 1);
  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;
  const int pp = threadIdx.x;                                            // pixel inside the tile = TMEM lane

  // weights -> bf16 hi / lo K-major operand (element (n = co, k) at (co/8)*2048 + (k/8)*128 + (co%8)*16 + (k%8)*2)
  for (int i = threadIdx.x; i < 32 * kHtKP; i += kHeadThreads) {
    const int co = i / kHtKP, k = i % kHtKP;
    const float v = (co < Co && k < K) ? __ldg(p.w + (size_t)co * K + k) : 0.f;
    const __nv_bfloat16 h = __float2bfloat16_rn(v);
    const __nv_bfloat16 l = __float2bfloat16_rn(v - __bfloat162float(h));
    const int off = (co >> 3) * kHtSbo + (k >> 3) * 128 + (co & 7) * 16 + (k & 7) * 2;
    *reinterpret_cast<__nv_bfloat16*>(s_w + off) = h;
    *reinterpret_cast<__nv_bfloat16*>(s_w + kHtWPart + off) = l;
  }
  if (threadIdx.x == 0) { mbar_init(s_bar, 1); fence_barrier_init(); }
  if (warp == 0) tmem_alloc(s_tmem, 256);
  fence_proxy_async();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *s_tmem;
  const uint32_t t_row = tmem + ((uint32_t)(warp * 32) << 16);           // 4 warps = the 4 TMEM lane quarters
  constexpr uint32_t kA_hi = 0, kA_lo = 64, kD = 128;
  const uint32_t el = elect_one();
  const uint64_t b_desc = make_desc(smem_u32(s_w), 128, kHtSbo);
  constexpr uint32_t idesc64 = make_idesc(128, 64), idesc32 = make_idesc(128, 32);
  float bias[32];
#pragma unroll
  for (int c = 0; c < 32; ++c) bias[c] = (p.bias && c < Co) ? __ldg(p.bias + c) : 0.f;

  const long long n_tiles = (p.P + kHeadTile - 1) / kHeadTile;
  uint32_t phase = 0;
  for (long long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const long long p0 = tile * kHeadTile;
    const int np = (int)((p.P - p0) < kHeadTile ? (p.P - p0) : kHeadTile);
    // ---- stage the tile's rows (contiguous spans of both sources): 8-byte cp.async, everything in flight at once (a
    //      register-staged loop kept ~4 KB per CTA in flight and made the kernel latency bound: 0.34 ms)
#pragma unroll 1
    for (int src = 0; src < 2; ++src) {
      const float* __restrict__ x = (src == 0 ? p.xa : p.xb);
      const int Cs = src == 0 ? p.Ca : p.Cb, k0 = src == 0 ? 0 : p.Ca;
      const int half = Cs >> 1;
      if (half == 0) continue;
      const float inv_half = 1.f / (float)half;
      const float2* __restrict__ x2 = reinterpret_cast<const float2*>(x + p0 * Cs);
#pragma unroll 4
      for (int i = threadIdx.x; i < np * half; i += kHeadThreads) {
        const int r = __float2int_rd(((float)i + 0.5f) * inv_half), k = (i - r * half) * 2;
        cp_async8(s_x + r * KS + k0 + k, x2 + i);
      }
    }
    cp_async_wait_all();
    __syncthreads();
    // ---- this pixel's row -> packed bf16 hi / lo pairs in tensor memory (8 packed columns per 16 k)
    {
      const float* __restrict__ xr = s_x + pp * KS;
      const bool row_ok = pp < np;
#pragma unroll 1
      for (int c8 = 0; c8 < kHtKP / 16; ++c8) {
        uint32_t hi[8], lo[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) {
          const int k = c8 * 16 + 2 * e;
          const float a = (row_ok && k < K) ? xr[k] : 0.f;
          const float b = (row_ok && k + 1 < K) ? xr[k + 1] : 0.f;
          split2(a, b, hi[e], lo[e]);
        }
        tmem_st8_issue(t_row + kA_hi + c8 * 8, hi);
        tmem_st8_issue(t_row + kA_lo + c8 * 8, lo);
      }
      tmem_st_wait();
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) {
      tc_fence_after();
#pragma unroll
      for (int kk = 0; kk < kHtKP / 16; ++kk) {
        const uint32_t ko = (kk * 256) >> 4;
        umma_bf16_ts_e(el, tmem + kD, tmem + kA_hi + kk * 8, b_desc + ko, idesc64, kk > 0 ? 1u : 0u);   // a_hi x [w_hi ; w_lo]
        umma_bf16_ts_e(el, tmem + kD, tmem + kA_lo + kk * 8, b_desc + ko, idesc32, 1u);                  // a_lo x w_hi
      }
      umma_commit_e(el, s_bar);
    }
    mbar_wait(s_bar, phase);
    phase ^= 1u;
    tc_fence_after();
    uint32_t d0[32], d1[32];
    tmem_ld32_issue(t_row + kD, d0);
    tmem_ld32_issue(t_row + kD + 32, d1);
    tmem_ld32_wait(d0);
    tmem_ld32_wait(d1);
    if (pp < np) {
      const long long pix = p0 + pp;
      const long long n = pix / p.HW, hw = pix - n * p.HW;
#pragma unroll
      for (int c = 0; c < 32; ++c) {
        if (c >= Co) break;
        const float v = __uint_as_float(d0[c]) + __uint_as_float(d1[c]) + bias[c];
        if (c < p.Co0) p.out0[(n * p.Co0 + c) * p.HW + hw] = v;
        else p.out1[(n * p.Co1 + (c - p.Co0)) * p.HW + hw] = v;
      }
    }
    tc_fence_before();      // the next tile's tcgen05.st / MMAs follow the __syncthreads after its staging loop
  }
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem, 256);
}

struct HeadsBwdParams {
  const float* g0; const float* g1;   // NCHW output gradients [n][Co0][HW], [n][Co1][HW]  (either may be NULL = zero)
  int Co0, Co1;
  const float* w;                     // [Co][Ca + Cb]
  float* ga; float* gb;               // NHWC source gradients [P][Ca], [P][Cb]  (either may be NULL = not needed)
  int Ca, Cb;
  long long P; int HW;
};

// one thread = one pixel of a 128-pixel tile: its output gradient (<= 32 values) lives in registers, the source gradient
// is produced four channels at a time (one broadcast LDS.128 of W[co][k..k+3] per four FMAs), staged in shared memory
// with an odd row stride and written out as the contiguous span it is (coalesced 8-byte stores)
template <int COP>
__global__ void __launch_bounds__(kHeadThreads) pixel_heads_bwd_kernel(const HeadsBwdParams p) {
  extern __shared__ __align__(16) float s_buf[];
  const int K = p.Ca + p.Cb, Co = p.Co0 + p.Co1;
  const int Kp = (K + 3) & ~3, KS = Kp | 1;
  float* s_w = s_buf;                            // [COP][Kp]
  float* s_o = s_buf + COP * Kp;                 // [kHeadTile][KS]
  for (int i = threadIdx.x; i < COP * Kp; i += blockDim.x) {
    const int c = i / Kp, k = i % Kp;
    s_w[i] = (c < Co && k < K) ? __ldg(p.w + (size_t)c * K + k) : 0.f;
  }
  const long long n_tiles = (p.P + kHeadTile - 1) / kHeadTile;
  for (long long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const long long p0 = tile * kHeadTile;
    const int np = (int)((p.P - p0) < kHeadTile ? (p.P - p0) : kHeadTile);
    __syncthreads();
    if ((int)threadIdx.x < np) {
      const long long pix = p0 + threadIdx.x;
      const long long n = pix / p.HW, hw = pix - n * p.HW;
      float g[COP];
#pragma unroll
      for (int c = 0; c < COP; ++c) {
        float v = 0.f;
        if (c < Co) {
          if (c < p.Co0) { if (p.g0) v = __ldg(p.g0 + (n * p.Co0 + c) * p.HW + hw); }
          else if (p.g1) v = __ldg(p.g1 + (n * p.Co1 + (c - p.Co0)) * p.HW + hw);
        }
        g[c] = v;
      }
      float* __restrict__ orow = s_o + threadIdx.x * KS;
#pragma unroll 2
      for (int k = 0; k < Kp; k += 4) {
        float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
#pragma unroll
        for (int c = 0; c < COP; ++c) {
          const float4 w = *reinterpret_cast<const float4*>(s_w + (size_t)c * Kp + k);
          a0 = fmaf(g[c], w.x, a0); a1 = fmaf(g[c], w.y, a1); a2 = fmaf(g[c], w.z, a2); a3 = fmaf(g[c], w.w, a3);
        }
        orow[k] = a0; orow[k + 1] = a1; orow[k + 2] = a2; orow[k + 3] = a3;
      }
    }
    __syncthreads();
#pragma unroll 1
    for (int src = 0; src < 2; ++src) {
      float* __restrict__ gx = src == 0 ? p.ga : p.gb;
      const int Cs = src == 0 ? p.Ca : p.Cb, k0 = src == 0 ? 0 : p.Ca;
      if (Cs == 0 || gx == nullptr) continue;
      const int half = Cs >> 1;
      float2* __restrict__ o2 = reinterpret_cast<float2*>(gx + p0 * Cs);
#pragma unroll 4
      for (int i = threadIdx.x; i < np * half; i += kHeadThreads) {
        const int pp = i / half, k = (i - pp * half) * 2;
        o2[i] = make_float2(s_o[pp * KS + k0 + k], s_o[pp * KS + k0 + k + 1]);
      }
    }
  }
}


// ---- tensor-core source gradient of the heads: [128 pixels x 32] x [32 x K]: the pixel's output gradient (read from the
// NCHW planes: coalesced) is the A operand in tensor memory, the stacked weights a K-major [N = k][K = co] B operand;
// the accumulator row (K columns) goes through shared memory to the NHWC rows with coalesced 8-byte stores.
constexpr int kHbSbo = (32 / 8) * 128;           // 512: byte stride between 8-row groups of the [128 k][32 co] operand
constexpr int kHbWPart = 16 * kHbSbo;            // 8192 bytes per part

__global__ void __launch_bounds__(kHeadThreads) pixel_heads_bwd_tc_kernel(const HeadsBwdParams p) {
  extern __shared__ __align__(16) unsigned char smem_raw_h[];
  unsigned char* sm = smem_raw_h + ((128u - (smem_u32(smem_raw_h) & 127u)) & 127u);
  const int K = p.Ca + p.Cb, Co = p.Co0 + p.Co1;
  const int KS = K;
  unsigned char* s_w = sm;                                               // W_hi | W_lo, [128 k][32 co] K-major
  float* s_o = reinterpret_cast<float*>(sm + 2 * kHbWPart);              // [kHeadTile][KS]
  uint64_t* s_bar = reinterpret_cast<uint64_t*>((reinterpret_cast<uintptr_t>(s_o + kHeadTile * KS) + 7) & ~uintptr_t(7));
  uint32_t* s_tmem = reinterpret_cast<uint32_t*>(s_bar + 1);
  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0);
  const int pp = threadIdx.x;

  for (int i = threadIdx.x; i < kHtKP * 32; i += kHeadThreads) {
    const int k = i >> 5, co = i & 31;
    const float v = (co < Co && k < K) ? __ldg(p.w + (size_t)co * K + k) : 0.f;
    const __nv_bfloat16 h = __float2bfloat16_rn(v);
    const __nv_bfloat16 l = __float2bfloat16_rn(v - __bfloat162float(h));
    const int off = (k >> 3) * kHbSbo + (co >> 3) * 128 + (k & 7) * 16 + (co & 7) * 2;
    *reinterpret_cast<__nv_bfloat16*>(s_w + off) = h;
    *reinterpret_cast<__nv_bfloat16*>(s_w + kHbWPart + off) = l;
  }
  if (threadIdx.x == 0) { mbar_init(s_bar, 1); fence_barrier_init(); }
  if (warp == 0) tmem_alloc(s_tmem, 256);
  fence_proxy_async();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *s_tmem;
  const uint32_t t_row = tmem + ((uint32_t)(warp * 32) << 16);
  constexpr uint32_t kA_hi = 0, kA_lo = 16, kD = 32;
  const uint32_t el = elect_one();
  const uint64_t b_hi = make_desc(smem_u32(s_w), 128, kHbSbo), b_lo = make_desc(smem_u32(s_w + kHbWPart), 128, kHbSbo);
  constexpr uint32_t idesc = make_idesc(128, kHtKP);

  const long long n_tiles = (p.P + kHeadTile - 1) / kHeadTile;
  uint32_t phase = 0;
  for (long long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const long long p0 = tile * kHeadTile;
    const int np = (int)((p.P - p0) < kHeadTile ? (p.P - p0) : kHeadTile);
    // ---- this pixel's output gradient -> packed bf16 hi / lo pairs in tensor memory
    {
      const long long pix = p0 + pp;
      const long long n = pix / p.HW, hw = pix - n * p.HW;
      float g[32];
#pragma unroll
      for (int c = 0; c < 32; ++c) {
        float v = 0.f;
        if (pp < np && c < Co) {
          if (c < p.Co0) { if (p.g0) v = __ldg(p.g0 + (n * p.Co0 + c) * p.HW + hw); }
          else if (p.g1) v = __ldg(p.g1 + (n * p.Co1 + (c - p.Co0)) * p.HW + hw);
        }
        g[c] = v;
      }
      uint32_t hi[16], lo[16];
#pragma unroll
      for (int e = 0; e < 16; ++e) split2(g[2 * e], g[2 * e + 1], hi[e], lo[e]);
      tmem_st16_issue(t_row + kA_hi, hi);
      tmem_st16_issue(t_row + kA_lo, lo);
      tmem_st_wait();
    }
    tc_fence_before();
    __syncthreads();           // also: the previous tile's copy-out of s_o is complete
    if (warp == 0) {
      tc_fence_after();
#pragma unroll
      for (int kk = 0; kk < 2; ++kk) {
        const uint32_t ko = (kk * 256) >> 4;
        umma_bf16_ts_e(el, tmem + kD, tmem + kA_hi + kk * 8, b_hi + ko, idesc, kk > 0 ? 1u : 0u);
        umma_bf16_ts_e(el, tmem + kD, tmem + kA_hi + kk * 8, b_lo + ko, idesc, 1u);
        umma_bf16_ts_e(el, tmem + kD, tmem + kA_lo + kk * 8, b_hi + ko, idesc, 1u);
      }
      umma_commit_e(el, s_bar);
    }
    mbar_wait(s_bar, phase);
    phase ^= 1u;
    tc_fence_after();
    {
      float* __restrict__ orow = s_o + pp * KS;
#pragma unroll 1
      for (int c = 0; c < 4; ++c) {
        uint32_t d[32];
        tmem_ld32_issue(t_row + kD + c * 32, d);
        tmem_ld32_wait(d);
#pragma unroll
        for (int i = 0; i < 32; ++i)
          if (c * 32 + i < K) orow[c * 32 + i] = __uint_as_float(d[i]);
      }
    }
    tc_fence_before();
    __syncthreads();
#pragma unroll 1
    for (int src = 0; src < 2; ++src) {
      float* __restrict__ gx = src == 0 ? p.ga : p.gb;
      const int Cs = src == 0 ? p.Ca : p.Cb, k0 = src == 0 ? 0 : p.Ca;
      if (Cs == 0 || gx == nullptr) continue;
      const int half = Cs >> 1;
      const float inv_half = 1.f / (float)half;
      float2* __restrict__ o2 = reinterpret_cast<float2*>(gx + p0 * Cs);
#pragma unroll 4
      for (int i = threadIdx.x; i < np * half; i += kHeadThreads) {
        const int r = __float2int_rd(((float)i + 0.5f) * inv_half), k = (i - r * half) * 2;
        o2[i] = *reinterpret_cast<const float2*>(s_o + r * KS + k0 + k);
      }
    }
  }
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem, 256);
}

// Weight / bias gradient of the stacked heads: dW[co][k] = sum_p g[co][p] x[p][k], db[co] = sum_p g[co][p].
// Each CTA reduces a strided set of 64-pixel tiles staged in shared memory (g transposed to [p][co], x as [p][k]); a thread
// owns a 4 (co) x 4 (k) register tile: per pixel one broadcast LDS.128 of g and one LDS.128 of x feed 16 FMAs.  Partials
// per CTA go to the workspace and are summed in a fixed order by column_reduce_kernel (deterministic).
constexpr int kWgTile = 64;
constexpr int kWgThreads = 256;

template <int COP>
__global__ void __launch_bounds__(kWgThreads) pixel_heads_wgrad_kernel(const HeadsBwdParams p, const float* __restrict__ xa, const float* __restrict__ xb,
                                                                      float* __restrict__ partial) {
  extern __shared__ __align__(16) float s_buf[];
  const int K = p.Ca + p.Cb, Co = p.Co0 + p.Co1;
  const int KG = (K + 3) >> 2, Kp = KG * 4;
  float* s_x = s_buf;                       // [kWgTile][Kp]
  float* s_g = s_buf + kWgTile * Kp;        // [kWgTile][COP]
  const int tid = threadIdx.x;
  const int kg = tid % KG, cog = tid / KG;
  const bool worker = cog < COP / 4;
  float acc[4][4], accb[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) { accb[i] = 0.f;
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f; }
  // zero the K padding columns once
  for (int i = tid; i < kWgTile * (Kp - K); i += kWgThreads) s_x[(i / (Kp - K)) * Kp + K + i % (Kp - K)] = 0.f;
  const long long n_tiles = (p.P + kWgTile - 1) / kWgTile;
  for (long long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const long long p0 = tile * kWgTile;
    const int np = (int)((p.P - p0) < kWgTile ? (p.P - p0) : kWgTile);
    __syncthreads();
    // x tile: both sources are contiguous [pixels][Cs] spans, copied with 8-byte cp.async (all in flight at once)
    for (int src = 0; src < 2; ++src) {
      const float* __restrict__ x = src == 0 ? xa : xb;
      const int Cs = src == 0 ? p.Ca : p.Cb, k0 = src == 0 ? 0 : p.Ca;
      const int half = Cs >> 1;
      if (half == 0) continue;
      const float inv_half = 1.f / (float)half;
      const float2* __restrict__ x2 = reinterpret_cast<const float2*>(x + p0 * Cs);
      for (int i = tid; i < kWgTile * half; i += kWgThreads) {
        const int pp = __float2int_rd(((float)i + 0.5f) * inv_half), k = (i - pp * half) * 2;
        if (pp < np) cp_async8(s_x + pp * Kp + k0 + k, x2 + i);
        else *reinterpret_cast<float2*>(s_x + pp * Kp + k0 + k) = make_float2(0.f, 0.f);
      }
    }
    // g tile, transposed: lanes run along the pixels (coalesced plane reads)
    for (int i = tid; i < COP * kWgTile; i += kWgThreads) {
      const int c = i / kWgTile, pp = i % kWgTile;
      float v = 0.f;
      if (pp < np && c < Co) {
        const long long pix = p0 + pp;
        const long long n = pix / p.HW, hw = pix - n * p.HW;
        if (c < p.Co0) { if (p.g0) v = __ldg(p.g0 + (n * p.Co0 + c) * p.HW + hw); }
        else if (p.g1) v = __ldg(p.g1 + (n * p.Co1 + (c - p.Co0)) * p.HW + hw);
      }
      s_g[pp * COP + c] = v;
    }
    cp_async_wait_all();
    __syncthreads();
    if (worker) {
#pragma unroll 4
      for (int pp = 0; pp < kWgTile; ++pp) {
        const float4 g = *reinterpret_cast<const float4*>(s_g + pp * COP + cog * 4);
        const float4 x = *reinterpret_cast<const float4*>(s_x + pp * Kp + kg * 4);
        const float gv[4] = {g.x, g.y, g.z, g.w}, xv[4] = {x.x, x.y, x.z, x.w};
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          accb[i] += gv[i];
#pragma unroll
          for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(gv[i], xv[j], acc[i][j]);
        }
      }
    }
  }
  if (worker) {
    float* row = partial + (size_t)blockIdx.x * (Co * K + Co);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int c = cog * 4 + i;
      if (c >= Co) continue;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int k = kg * 4 + j;
        if (k < K) row[c * K + k] = acc[i][j];
      }
      if (kg == 0) row[Co * K + c] = accb[i];
    }
  }
}

// ---- tensor-core weight / bias gradient of the heads: D[k][co] += sum_pixels x[pixel][k] g[pixel][co], accumulated in
// tensor memory over ALL tiles of the (persistent) CTA.  A = x^T: TMEM lane = source channel k, a tile's 128 pixels are
// the reduction dimension (thread k reads column k of the staged tile: conflict free); row K of A is all ones, so row K
// of D is the bias gradient.  B = g^T [N = co][K = pixels], bf16 hi / lo K-major in shared memory, rebuilt per tile by
// the thread that owns the pixel.  Per-CTA partials go to the workspace, summed in fixed order by column_reduce_kernel.
__global__ void __launch_bounds__(kHeadThreads) pixel_heads_wgrad_tc_kernel(const HeadsBwdParams p, const float* __restrict__ xa,
                                                                          const float* __restrict__ xb, float* __restrict__ partial) {
  extern __shared__ __align__(16) unsigned char smem_raw_h[];
  unsigned char* sm = smem_raw_h + ((128u - (smem_u32(smem_raw_h) & 127u)) & 127u);
  const int K = p.Ca + p.Cb, Co = p.Co0 + p.Co1;
  const int KS = K;
  unsigned char* s_g = sm;                                               // [G_hi ; G_lo], [32 co][128 pixels] K-major
  float* s_x = reinterpret_cast<float*>(sm + 2 * kHtWPart);              // [kHeadTile][KS]
  uint64_t* s_bar = reinterpret_cast<uint64_t*>((reinterpret_cast<uintptr_t>(s_x + kHeadTile * KS) + 7) & ~uintptr_t(7));
  uint32_t* s_tmem = reinterpret_cast<uint32_t*>(s_bar + 1);
  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0);
  const int t = threadIdx.x;                      // pixel of the tile when building B, source channel k when building A

  for (int i = threadIdx.x; i < (2 * kHtWPart) / 4; i += kHeadThreads) reinterpret_cast<uint32_t*>(s_g)[i] = 0u;
  if (threadIdx.x == 0) { mbar_init(s_bar, 1); fence_barrier_init(); }
  if (warp == 0) tmem_alloc(s_tmem, 256);
  fence_proxy_async();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *s_tmem;
  const uint32_t t_row = tmem + ((uint32_t)(warp * 32) << 16);
  constexpr uint32_t kA_hi = 0, kA_lo = 64, kD = 128;
  const uint32_t el = elect_one();
  const uint64_t b_desc = make_desc(smem_u32(s_g), 128, kHtSbo);
  constexpr uint32_t idesc64 = make_idesc(128, 64), idesc32 = make_idesc(128, 32);
  const int b_off = (t >> 3) * 128 + (t & 7) * 2;          // this pixel's slot inside each 8-row group of the B operand

  const long long n_tiles = (p.P + kHeadTile - 1) / kHeadTile;
  int done = 0;
  for (long long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++done) {
    const long long p0 = tile * kHeadTile;
    const int np = (int)((p.P - p0) < kHeadTile ? (p.P - p0) : kHeadTile);
    // ---- x tile -> shared memory (the previous tile's readers finished before its MMAs were issued)
#pragma unroll 1
    for (int src = 0; src < 2; ++src) {
      const float* __restrict__ x = src == 0 ? xa : xb;
      const int Cs = src == 0 ? p.Ca : p.Cb, k0 = src == 0 ? 0 : p.Ca;
      const int half = Cs >> 1;
      if (half == 0) continue;
      const float inv_half = 1.f / (float)half;
      const float2* __restrict__ x2 = reinterpret_cast<const float2*>(x + p0 * Cs);
#pragma unroll 4
      for (int i = threadIdx.x; i < np * half; i += kHeadThreads) {
        const int r = __float2int_rd(((float)i + 0.5f) * inv_half), k = (i - r * half) * 2;
        cp_async8(s_x + r * KS + k0 + k, x2 + i);
      }
    }
    // ---- this pixel's output gradient (NCHW planes: coalesced)
    float g[32];
    {
      const long long pix = p0 + t;
      const long long n = pix / p.HW, hw = pix - n * p.HW;
#pragma unroll
      for (int c = 0; c < 32; ++c) {
        float v = 0.f;
        if (t < np && c < Co) {
          if (c < p.Co0) { if (p.g0) v = __ldg(p.g0 + (n * p.Co0 + c) * p.HW + hw); }
          else if (p.g1) v = __ldg(p.g1 + (n * p.Co1 + (c - p.Co0)) * p.HW + hw);
        }
        g[c] = v;
      }
    }
    // the previous tile's MMAs must be done with the B operand and the A columns before either is rewritten
    if (done > 0) { mbar_wait(s_bar, (done - 1) & 1); tc_fence_after(); }
#pragma unroll
    for (int c = 0; c < 32; ++c) {
      const __nv_bfloat16 h = __float2bfloat16_rn(g[c]);
      const __nv_bfloat16 l = __float2bfloat16_rn(g[c] - __bfloat162float(h));
      const int off = (c >> 3) * kHtSbo + (c & 7) * 16 + b_off;
      *reinterpret_cast<__nv_bfloat16*>(s_g + off) = h;
      *reinterpret_cast<__nv_bfloat16*>(s_g + kHtWPart + off) = l;
    }
    cp_async_wait_all();
    fence_proxy_async();
    __syncthreads();
    // ---- column t of the tile (source channel t over the 128 pixels) -> packed bf16 hi / lo pairs in tensor memory
    {
      const int k = t;
#pragma unroll 1
      for (int c8 = 0; c8 < kHeadTile / 16; ++c8) {
        uint32_t hi[8], lo[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) {
          const int r0 = c8 * 16 + 2 * e;
          float a = 0.f, b = 0.f;
          if (k < K) { a = r0 < np ? s_x[r0 * KS + k] : 0.f; b = r0 + 1 < np ? s_x[(r0 + 1) * KS + k] : 0.f; }
          else if (k == K) { a = r0 < np ? 1.f : 0.f; b = r0 + 1 < np ? 1.f : 0.f; }     // ones row: bias gradient
          split2(a, b, hi[e], lo[e]);
        }
        tmem_st8_issue(t_row + kA_hi + c8 * 8, hi);
        tmem_st8_issue(t_row + kA_lo + c8 * 8, lo);
      }
      tmem_st_wait();
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) {
      tc_fence_after();
#pragma unroll
      for (int kk = 0; kk < kHeadTile / 16; ++kk) {
        const uint32_t ko = (kk * 256) >> 4;
        const uint32_t acc = (done > 0 || kk > 0) ? 1u : 0u;
        umma_bf16_ts_e(el, tmem + kD, tmem + kA_hi + kk * 8, b_desc + ko, idesc64, acc);       // x_hi x [g_hi ; g_lo]
        umma_bf16_ts_e(el, tmem + kD, tmem + kA_lo + kk * 8, b_desc + ko, idesc32, 1u);        // x_lo x g_hi
      }
      umma_commit_e(el, s_bar);
    }
  }
  if (done > 0) { mbar_wait(s_bar, (done - 1) & 1); tc_fence_after(); }
  uint32_t d0[32], d1[32];
  tmem_ld32_issue(t_row + kD, d0);
  tmem_ld32_issue(t_row + kD + 32, d1);
  tmem_ld32_wait(d0);
  tmem_ld32_wait(d1);
  if (t <= K) {
    float* row = partial + (size_t)blockIdx.x * (Co * K + Co);
#pragma unroll
    for (int c = 0; c < 32; ++c) {
      if (c >= Co) break;
      const float v = done > 0 ? __uint_as_float(d0[c]) + __uint_as_float(d1[c]) : 0.f;
      if (t < K) row[c * K + t] = v;
      else row[Co * K + c] = v;
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem, 256);
}

int heads_check(int Ca, int Cb, int Co0, int Co1, long long P, int HW) {
  ISA_CHECK_ARG(Ca > 0 && Cb >= 0 && Ca % 2 == 0 && Cb % 2 == 0, "pixel_heads: source widths must be even (Ca=%d Cb=%d)", Ca, Cb);
  ISA_CHECK_ARG(Co0 > 0 && Co1 >= 0 && Co0 + Co1 <= 32, "pixel_heads: at most 32 stacked output channels (Co0=%d Co1=%d)", Co0, Co1);
  ISA_CHECK_ARG(P > 0 && HW > 0 && P % HW == 0, "pixel_heads: P=%lld must be a multiple of HW=%d", P, HW);
  ISA_CHECK_ARG((size_t)(Ca + Cb + 4) * (32 + kHeadTile + 1) * sizeof(float) <= 200 * 1024, "pixel_heads: Ca + Cb = %d too wide for the shared-memory tiles", Ca + Cb);
  return ISA_OK;
}

}  // namespace

extern "C" {

// Workspace of isa_bias_act_bwd: per-CTA partial column sums.
size_t isa_bias_act_workspace_bytes(int C) {
  if (C <= 0) return 0;
  IsaDeviceInfo di;
  if (isa_device_info(&di)) return 0;
  return (size_t)di.num_sms * 8 * C * sizeof(float);
}

// x [rows][C] (NHWC activation) <- act(x + bias[c]) in place; relu != 0 selects max(.,0).  1 <= C <= 256.
int isa_bias_act_fwd(float* x, const float* bias, long long rows, int C, int relu, cudaStream_t stream) {
  ISA_CHECK_ARG(x && bias && rows > 0 && C > 0 && C <= kThreads, "bias_act_fwd: bad argument (rows=%lld C=%d)", rows, C);
  IsaDeviceInfo di;
  int rc = isa_device_info(&di);
  if (rc) return rc;
  const bool v4 = (C % 4 == 0) && ((uintptr_t)x % 16 == 0);
  const int grid = bias_act_grid(rows, C, v4 ? 4 : 1, di.num_sms);
  if (v4) {
    if (relu) bias_act_fwd_kernel<4, true><<<grid, kThreads, 0, stream>>>(x, bias, rows, C);
    else bias_act_fwd_kernel<4, false><<<grid, kThreads, 0, stream>>>(x, bias, rows, C);
  } else {
    if (relu) bias_act_fwd_kernel<1, true><<<grid, kThreads, 0, stream>>>(x, bias, rows, C);
    else bias_act_fwd_kernel<1, false><<<grid, kThreads, 0, stream>>>(x, bias, rows, C);
  }
  ISA_CUDA(cudaGetLastError());
  return ISA_OK;
}

// gx = relu ? gy * (y > 0) : gy  (gx may be NULL without relu: nothing to write; gx may alias gy);  dbias[c] = sum_r gx[r][c].
// y is the forward output (only read with relu).  workspace: isa_bias_act_workspace_bytes(C).
int isa_bias_act_bwd(const float* gy, const float* y, float* gx, float* dbias, long long rows, int C, int relu, void* workspace,
                     size_t workspace_bytes, cudaStream_t stream) {
  ISA_CHECK_ARG(gy && dbias && rows > 0 && C > 0 && C <= kThreads && workspace, "bias_act_bwd: bad argument (rows=%lld C=%d)", rows, C);
  ISA_CHECK_ARG(!relu || (y && gx), "bias_act_bwd: relu needs the forward output and a gradient buffer");
  if (workspace_bytes < isa_bias_act_workspace_bytes(C)) {
    isa_set_error("bias_act_bwd: workspace too small");
    return ISA_ERR_WORKSPACE;
  }
  IsaDeviceInfo di;
  int rc = isa_device_info(&di);
  if (rc) return rc;
  const bool v4 = (C % 4 == 0) && ((uintptr_t)gy % 16 == 0) && (!y || (uintptr_t)y % 16 == 0) && (!gx || (uintptr_t)gx % 16 == 0);
  const int grid = bias_act_grid(rows, C, v4 ? 4 : 1, di.num_sms);
  float* partial = reinterpret_cast<float*>(workspace);
  if (v4) {
    if (relu) bias_act_bwd_kernel<4, true><<<grid, kThreads, 0, stream>>>(gy, y, gx, partial, rows, C);
    else bias_act_bwd_kernel<4, false><<<grid, kThreads, 0, stream>>>(gy, y, gx, partial, rows, C);
  } else {
    if (relu) bias_act_bwd_kernel<1, true><<<grid, kThreads, 0, stream>>>(gy, y, gx, partial, rows, C);
    else bias_act_bwd_kernel<1, false><<<grid, kThreads, 0, stream>>>(gy, y, gx, partial, rows, C);
  }
  ISA_CUDA(cudaGetLastError());
  column_reduce_kernel<<<(C + 31) / 32, 256, 0, stream>>>(partial, grid, C, dbias);
  ISA_CUDA(cudaGetLastError());
  return ISA_OK;
}

// Workspace of isa_add_layernorm_bwd.
size_t isa_add_layernorm_workspace_bytes(long long rows, int C) {
  if (rows <= 0 || C <= 0) return 0;
  const size_t grid = (size_t)((rows + kThreads - 1) / kThreads);
  return (grid + 1) * 2 * C * sizeof(float);
}

// y = LayerNorm(x + res) * gamma + beta over the last dimension C (biased variance, like nn.LayerNorm); res may be NULL.
// stats [rows][2] receives (mean, rstd) for the backward.  C in {8,16,24,32,40,48,64}.
int isa_add_layernorm_fwd(const float* x, const float* res, const float* gamma, const float* beta, long long rows, int C, float eps, float* y,
                          float* stats, cudaStream_t stream) {
  ISA_CHECK_ARG(x && gamma && beta && y && stats && rows > 0, "add_layernorm_fwd: bad argument");
  if (!ln_width_ok(C)) {
    isa_set_error("add_layernorm: width %d not in {8,16,24,32,40,48,64}", C);
    return ISA_ERR_UNSUPPORTED;
  }
  switch (C) {
    case 8: return launch_ln_fwd<8>(x, res, gamma, beta, rows, eps, y, stats, stream);
    case 16: return launch_ln_fwd<16>(x, res, gamma, beta, rows, eps, y, stats, stream);
    case 24: return launch_ln_fwd<24>(x, res, gamma, beta, rows, eps, y, stats, stream);
    case 32: return launch_ln_fwd<32>(x, res, gamma, beta, rows, eps, y, stats, stream);
    case 40: return launch_ln_fwd<40>(x, res, gamma, beta, rows, eps, y, stats, stream);
    case 48: return launch_ln_fwd<48>(x, res, gamma, beta, rows, eps, y, stats, stream);
    default: return launch_ln_fwd<64>(x, res, gamma, beta, rows, eps, y, stats, stream);
  }
}

// gv = d loss / d (x + res) (the gradient of both summands), dgamma, dbeta [C].
int isa_add_layernorm_bwd(const float* gy, const float* x, const float* res, const float* gamma, const float* stats, long long rows, int C,
                          float* gv, float* dgamma, float* dbeta, void* workspace, size_t workspace_bytes, cudaStream_t stream) {
  ISA_CHECK_ARG(gy && x && gamma && stats && gv && dgamma && dbeta && workspace && rows > 0, "add_layernorm_bwd: bad argument");
  if (!ln_width_ok(C)) {
    isa_set_error("add_layernorm: width %d not in {8,16,24,32,40,48,64}", C);
    return ISA_ERR_UNSUPPORTED;
  }
  if (workspace_bytes < isa_add_layernorm_workspace_bytes(rows, C)) {
    isa_set_error("add_layernorm_bwd: workspace too small");
    return ISA_ERR_WORKSPACE;
  }
  float* partial = reinterpret_cast<float*>(workspace);
  switch (C) {
    case 8: return launch_ln_bwd<8>(gy, x, res, gamma, stats, rows, gv, dgamma, dbeta, partial, stream);
    case 16: return launch_ln_bwd<16>(gy, x, res, gamma, stats, rows, gv, dgamma, dbeta, partial, stream);
    case 24: return launch_ln_bwd<24>(gy, x, res, gamma, stats, rows, gv, dgamma, dbeta, partial, stream);
    case 32: return launch_ln_bwd<32>(gy, x, res, gamma, stats, rows, gv, dgamma, dbeta, partial, stream);
    case 40: return launch_ln_bwd<40>(gy, x, res, gamma, stats, rows, gv, dgamma, dbeta, partial, stream);
    case 48: return launch_ln_bwd<48>(gy, x, res, gamma, stats, rows, gv, dgamma, dbeta, partial, stream);
    default: return launch_ln_bwd<64>(gy, x, res, gamma, stats, rows, gv, dgamma, dbeta, partial, stream);
  }
}

// out0 [n][Co0][HW], out1 [n][Co1][HW] (NCHW planes) = stacked 1x1 convolution w [Co0+Co1][Ca+Cb] (+ bias) of the
// channel concatenation of the NHWC sources xa [P][Ca], xb [P][Cb]; P = n * HW pixels; Ca, Cb even; Co0 + Co1 <= 32.
int isa_pixel_heads_fwd(const float* xa, int Ca, const float* xb, int Cb, const float* w, const float* bias, float* out0, int Co0,
                        float* out1, int Co1, long long P, int HW, cudaStream_t stream) {
  int rc = heads_check(Ca, Cb, Co0, Co1, P, HW);
  if (rc) return rc;
  ISA_CHECK_ARG(xa && (xb || Cb == 0) && w && out0 && (out1 || Co1 == 0), "pixel_heads_fwd: null pointer");
  IsaDeviceInfo di;
  rc = isa_device_info(&di);
  if (rc) return rc;
  HeadsParams hp;
  hp.xa = xa; hp.xb = xb; hp.Ca = Ca; hp.Cb = Cb; hp.w = w; hp.bias = bias; hp.out0 = out0; hp.out1 = out1; hp.Co0 = Co0; hp.Co1 = Co1;
  hp.P = P; hp.HW = HW;
  const int Co = Co0 + Co1, cop = (Co + 3) & ~3;
  const long long n_tiles = (P + kHeadTile - 1) / kHeadTile;
  long long grid = n_tiles < (long long)di.num_sms * 3 ? n_tiles : (long long)di.num_sms * 3;
  if (Ca + Cb <= kHtKP) {
    // tensor-core path: 2 CTAs per SM (256 TMEM columns each)
    size_t smem = 2 * kHtWPart + (size_t)kHeadTile * (Ca + Cb) * sizeof(float) + 64 + 128;
    if (smem < 80 * 1024) smem = 80 * 1024;     // never three CTAs on one SM: the third would spin in tcgen05.alloc
    grid = n_tiles < (long long)di.num_sms * 2 ? n_tiles : (long long)di.num_sms * 2;
    ISA_CUDA(cudaFuncSetAttribute(pixel_heads_fwd_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    pixel_heads_fwd_tc_kernel<<<(unsigned)grid, kHeadThreads, smem, stream>>>(hp);
    ISA_CUDA(cudaGetLastError());
    return ISA_OK;
  }
#define ISA_HEADS_FWD(COP)                                                                                              \
  {                                                                                                                     \
    const size_t smem = ((size_t)(Ca + Cb) * COP + (size_t)kHeadTile * ((Ca + Cb) | 1)) * sizeof(float);                \
    ISA_CUDA(cudaFuncSetAttribute(pixel_heads_fwd_kernel<COP>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
    pixel_heads_fwd_kernel<COP><<<(unsigned)grid, kHeadThreads, smem, stream>>>(hp);                                    \
  }
  if (cop <= 4) ISA_HEADS_FWD(4)
  else if (cop <= 8) ISA_HEADS_FWD(8)
  else if (cop <= 16) ISA_HEADS_FWD(16)
  else if (cop <= 24) ISA_HEADS_FWD(24)
  else if (cop <= 28) ISA_HEADS_FWD(28)
  else ISA_HEADS_FWD(32)
#undef ISA_HEADS_FWD
  ISA_CUDA(cudaGetLastError());
  return ISA_OK;
}

// ga [P][Ca], gb [P][Cb] (NHWC; either may be NULL) = gradient of the sources given the NCHW output gradients g0, g1
// (either may be NULL = zero).  The weight / bias gradients are plain GEMMs / row sums left to the caller.
int isa_pixel_heads_bwd(const float* g0, int Co0, const float* g1, int Co1, const float* w, float* ga, int Ca, float* gb, int Cb,
                        long long P, int HW, cudaStream_t stream) {
  int rc = heads_check(Ca, Cb, Co0, Co1, P, HW);
  if (rc) return rc;
  ISA_CHECK_ARG(w && (ga || gb), "pixel_heads_bwd: null pointer");
  IsaDeviceInfo di;
  rc = isa_device_info(&di);
  if (rc) return rc;
  HeadsBwdParams hp;
  hp.g0 = g0; hp.g1 = g1; hp.Co0 = Co0; hp.Co1 = Co1; hp.w = w; hp.ga = ga; hp.gb = gb; hp.Ca = Ca; hp.Cb = Cb; hp.P = P; hp.HW = HW;
  const int Co = Co0 + Co1, cop = (Co + 3) & ~3;
  const long long n_tiles = (P + kHeadTile - 1) / kHeadTile;
  long long grid = n_tiles < (long long)di.num_sms * 3 ? n_tiles : (long long)di.num_sms * 3;
  const int Kp = (Ca + Cb + 3) & ~3;
  if (Ca + Cb <= kHtKP) {
    size_t smem = 2 * kHbWPart + (size_t)kHeadTile * (Ca + Cb) * sizeof(float) + 64 + 128;
    if (smem < 80 * 1024) smem = 80 * 1024;     // at most two CTAs per SM (256 TMEM columns each)
    grid = n_tiles < (long long)di.num_sms * 2 ? n_tiles : (long long)di.num_sms * 2;
    ISA_CUDA(cudaFuncSetAttribute(pixel_heads_bwd_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    pixel_heads_bwd_tc_kernel<<<(unsigned)grid, kHeadThreads, smem, stream>>>(hp);
    ISA_CUDA(cudaGetLastError());
    return ISA_OK;
  }
#define ISA_HEADS_BWD(COP)                                                                                              \
  {                                                                                                                     \
    const size_t smem = ((size_t)Kp * COP + (size_t)kHeadTile * (Kp | 1)) * sizeof(float);                              \
    ISA_CUDA(cudaFuncSetAttribute(pixel_heads_bwd_kernel<COP>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
    pixel_heads_bwd_kernel<COP><<<(unsigned)grid, kHeadThreads, smem, stream>>>(hp);                                    \
  }
  if (cop <= 4) ISA_HEADS_BWD(4)
  else if (cop <= 8) ISA_HEADS_BWD(8)
  else if (cop <= 16) ISA_HEADS_BWD(16)
  else if (cop <= 24) ISA_HEADS_BWD(24)
  else if (cop <= 28) ISA_HEADS_BWD(28)
  else ISA_HEADS_BWD(32)
#undef ISA_HEADS_BWD
  ISA_CUDA(cudaGetLastError());
  return ISA_OK;
}

// Workspace of isa_pixel_heads_wgrad.
size_t isa_pixel_heads_wgrad_workspace_bytes(int Ca, int Cb, int Co0, int Co1) {
  IsaDeviceInfo di;
  if (isa_device_info(&di)) return 0;
  return (size_t)di.num_sms * 2 * (size_t)((Co0 + Co1) * (Ca + Cb + 1)) * sizeof(float);
}

// dw [Co0+Co1][Ca+Cb] and db [Co0+Co1] (contiguous: dw then db in `dw_db`) from the NCHW output gradients and the NHWC
// sources; deterministic.  (Ca + Cb + 3) / 4 * ((Co0 + Co1 + 3) / 4) must be <= 256.
int isa_pixel_heads_wgrad(const float* g0, int Co0, const float* g1, int Co1, const float* xa, int Ca, const float* xb, int Cb,
                          long long P, int HW, float* dw_db, void* workspace, size_t workspace_bytes, cudaStream_t stream) {
  int rc = heads_check(Ca, Cb, Co0, Co1, P, HW);
  if (rc) return rc;
  ISA_CHECK_ARG(xa && (xb || Cb == 0) && dw_db && workspace && (g0 || g1), "pixel_heads_wgrad: null pointer");
  const int K = Ca + Cb, Co = Co0 + Co1, cop = (Co + 3) & ~3, KG = (K + 3) / 4;
  ISA_CHECK_ARG(KG * (cop / 4) <= kWgThreads, "pixel_heads_wgrad: %d x %d outputs exceed one CTA's register tiles", Co, K);
  if (workspace_bytes < isa_pixel_heads_wgrad_workspace_bytes(Ca, Cb, Co0, Co1)) {
    isa_set_error("pixel_heads_wgrad: workspace too small");
    return ISA_ERR_WORKSPACE;
  }
  IsaDeviceInfo di;
  rc = isa_device_info(&di);
  if (rc) return rc;
  HeadsBwdParams hp;
  hp.g0 = g0; hp.g1 = g1; hp.Co0 = Co0; hp.Co1 = Co1; hp.w = nullptr; hp.ga = nullptr; hp.gb = nullptr; hp.Ca = Ca; hp.Cb = Cb; hp.P = P; hp.HW = HW;
  const long long n_tiles = (P + kWgTile - 1) / kWgTile;
  const int grid = (int)(n_tiles < (long long)di.num_sms * 2 ? n_tiles : (long long)di.num_sms * 2);
  float* partial = reinterpret_cast<float*>(workspace);
  if (K + 1 <= kHtKP) {
    size_t smem = 2 * kHtWPart + (size_t)kHeadTile * K * sizeof(float) + 64 + 128;
    if (smem < 80 * 1024) smem = 80 * 1024;     // at most two CTAs per SM (256 TMEM columns each)
    const long long nt = (P + kHeadTile - 1) / kHeadTile;
    const int g2 = (int)(nt < (long long)di.num_sms * 2 ? nt : (long long)di.num_sms * 2);
    ISA_CUDA(cudaFuncSetAttribute(pixel_heads_wgrad_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    pixel_heads_wgrad_tc_kernel<<<g2, kHeadThreads, smem, stream>>>(hp, xa, xb, partial);
    ISA_CUDA(cudaGetLastError());
    const int R2 = Co * K + Co;
    column_reduce_kernel<<<(R2 + 31) / 32, 256, 0, stream>>>(partial, g2, R2, dw_db);
    ISA_CUDA(cudaGetLastError());
    return ISA_OK;
  }
#define ISA_HEADS_WG(COP)                                                                                                  \
  {                                                                                                                        \
    const size_t smem = (size_t)kWgTile * (KG * 4 + COP) * sizeof(float);                                                  \
    ISA_CUDA(cudaFuncSetAttribute(pixel_heads_wgrad_kernel<COP>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
    pixel_heads_wgrad_kernel<COP><<<grid, kWgThreads, smem, stream>>>(hp, xa, xb, partial);                                \
  }
  if (cop <= 4) ISA_HEADS_WG(4)
  else if (cop <= 8) ISA_HEADS_WG(8)
  else if (cop <= 16) ISA_HEADS_WG(16)
  else if (cop <= 24) ISA_HEADS_WG(24)
  else if (cop <= 28) ISA_HEADS_WG(28)
  else ISA_HEADS_WG(32)
#undef ISA_HEADS_WG
  ISA_CUDA(cudaGetLastError());
  const int R = Co * K + Co;
  column_reduce_kernel<<<(R + 31) / 32, 256, 0, stream>>>(partial, grid, R, dw_db);
  ISA_CUDA(cudaGetLastError());
  return ISA_OK;
}

// y [N][H/2][W/2][C] = 2x2 / stride-2 max pool of the NHWC tensor x [N][H][W][C] (floor mode; C % 4 == 0);
// idx (u8, same shape as y, may be NULL at inference) = window position 0..3 of the maximum.
int isa_maxpool2x2_fwd(const float* x, int N, int H, int W, int C, float* y, unsigned char* idx, cudaStream_t stream) {
  ISA_CHECK_ARG(x && y && N > 0 && H >= 2 && W >= 2 && C > 0 && C % 4 == 0, "maxpool2x2_fwd: bad argument (N=%d H=%d W=%d C=%d)", N, H, W, C);
  IsaDeviceInfo di;
  int rc = isa_device_info(&di);
  if (rc) return rc;
  const int Ho = H / 2, Wo = W / 2, C4 = C / 4;
  const long long total4 = (long long)N * Ho * Wo * C4;
  long long grid = (total4 + 255) / 256;
  if (grid > (long long)di.num_sms * 16) grid = (long long)di.num_sms * 16;
  maxpool2x2_fwd_kernel<<<(unsigned)grid, 256, 0, stream>>>(x, y, idx, total4, Ho, Wo, W, C4, (long long)H * W * C);
  ISA_CUDA(cudaGetLastError());
  return ISA_OK;
}

// gx [N][H][W][C] = scatter of gy [N][H/2][W/2][C] to the recorded window positions (every covered element is written;
// with odd H or W the uncovered last row / column is zeroed first).
int isa_maxpool2x2_bwd(const float* gy, const unsigned char* idx, int N, int H, int W, int C, const float* skip_grad,
                       long long skip_pixel_stride, float* gx, cudaStream_t stream) {
  ISA_CHECK_ARG(gy && idx && gx && N > 0 && H >= 2 && W >= 2 && C > 0 && C % 4 == 0, "maxpool2x2_bwd: bad argument (N=%d H=%d W=%d C=%d)", N, H, W, C);
  ISA_CHECK_ARG(!skip_grad || (!(H & 1) && !(W & 1) && skip_pixel_stride >= C && skip_pixel_stride % 4 == 0 &&
                               (reinterpret_cast<uintptr_t>(skip_grad) & 15u) == 0),
                "maxpool2x2_bwd: a skip gradient needs even H, W, a pixel stride >= C that is a multiple of 4 and 16-byte alignment");
  IsaDeviceInfo di;
  int rc = isa_device_info(&di);
  if (rc) return rc;
  if ((H & 1) || (W & 1)) ISA_CUDA(cudaMemsetAsync(gx, 0, (size_t)N * H * W * C * sizeof(float), stream));
  const int Ho = H / 2, Wo = W / 2, C4 = C / 4;
  const long long total4 = (long long)N * Ho * Wo * C4;
  long long grid = (total4 + 255) / 256;
  if (grid > (long long)di.num_sms * 16) grid = (long long)di.num_sms * 16;
  maxpool2x2_bwd_kernel<<<(unsigned)grid, 256, 0, stream>>>(gy, idx, gx, total4, Ho, Wo, W, C4, (long long)H * W * C, skip_grad, skip_pixel_stride);
  ISA_CUDA(cudaGetLastError());
  return ISA_OK;
}

// Workspace of isa_adadelta_step (per-CTA partial sums of squares).
size_t isa_adadelta_workspace_bytes(void) {
  IsaDeviceInfo di;
  if (isa_device_info(&di)) return 0;
  return (size_t)di.num_sms * 4 * sizeof(double);
}

// One optimizer step over flat fp32 buffers of n elements (16-byte aligned): optional global-norm clipping
// (max_norm > 0; coefficient min(1, max_norm / (norm + 1e-6)) like torch.nn.utils.clip_grad_norm_), then PyTorch's
// Adadelta update with L2 weight decay.  grad is read only; norm_out (device float, may be NULL) receives the norm.
int isa_adadelta_step(float* param, const float* grad, float* square_avg, float* acc_delta, long long n, float lr, float rho, float eps,
                      float weight_decay, float max_norm, float* norm_out, void* workspace, size_t workspace_bytes, cudaStream_t stream) {
  ISA_CHECK_ARG(param && grad && square_avg && acc_delta && n > 0 && workspace, "adadelta_step: bad argument");
  ISA_CHECK_ARG(((reinterpret_cast<uintptr_t>(param) | reinterpret_cast<uintptr_t>(grad) | reinterpret_cast<uintptr_t>(square_avg) |
                  reinterpret_cast<uintptr_t>(acc_delta)) & 15u) == 0, "adadelta_step: buffers must be 16-byte aligned");
  if (workspace_bytes < isa_adadelta_workspace_bytes()) {
    isa_set_error("adadelta_step: workspace too small");
    return ISA_ERR_WORKSPACE;
  }
  IsaDeviceInfo di;
  int rc = isa_device_info(&di);
  if (rc) return rc;
  long long grid = ((n >> 2) + 255) / 256;
  if (grid < 1) grid = 1;
  if (grid > (long long)di.num_sms * 4) grid = (long long)di.num_sms * 4;
  double* partial = reinterpret_cast<double*>(workspace);
  const bool need_norm = max_norm > 0.f || norm_out;
  if (need_norm) {
    sumsq_partial_kernel<<<(unsigned)grid, 256, 0, stream>>>(grad, n, partial);
    ISA_CUDA(cudaGetLastError());
  }
  AdadeltaParams a;
  a.param = param; a.grad = grad; a.square_avg = square_avg; a.acc_delta = acc_delta; a.n = n;
  a.lr = lr; a.rho = rho; a.eps = eps; a.weight_decay = weight_decay; a.max_norm = max_norm;
  a.partial = partial; a.n_partial = need_norm ? (int)grid : 0; a.norm_out = norm_out;
  adadelta_step_kernel<<<(unsigned)grid, 256, 0, stream>>>(a);
  ISA_CUDA(cudaGetLastError());
  return ISA_OK;
}

}  // extern "C"
