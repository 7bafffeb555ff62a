// Persistent bidirectional-GRU scan for the ReNet row / column sweeps.
//
// Reference contract: /root/reference/code/lib/archs/modules/README.md:225-256 (ReNet: a
// bidirectional GRU over every row, then over every column of the result; renet.py itself is
// absent from the tree, so the arithmetic is PyTorch's nn.GRU:
//     r = sigmoid(W_ir x + b_ir + W_hr h + b_hr)      z = sigmoid(W_iz x + b_iz + W_hz h + b_hz)
//     n = tanh(W_in x + b_in + r * (W_hn h + b_hn))   h' = (1 - z) * n + z * h
// with weight_hh_l0 laid out (3n, n) in gate order r, z, n).
//
// Split of the work: the input projection gx = x W_ih^T + b_ih is one big GEMM over all
// tokens (library GEMM on the host side); this kernel is the sequential part.  One CTA owns S
// sequences of ONE direction for the whole sweep:
//   * W_hh^T (n x 3n fp32, 120 KB for n = 100) is loaded into shared memory once and stays
//     there for all T steps; h_{t-1} of the S sequences lives in shared memory (double buffered);
//   * per step each thread owns one hidden unit j and S/2 sequences: 3 * S/2 fp32 accumulators
//     over i = 0..n-1 (W row reads are conflict free, h reads are warp broadcasts), then the
//     gate math in registers; the next step's gx values are prefetched into registers while the
//     current step computes;
//   * all tensors are token-major ("channels last"): a sequence's per-step chunk is contiguous,
//     so every global access of a warp is a full 128 B line.  Rows and columns differ only in
//     the token strides handed in.
// Backward (BPTT) walks the other way with W_hh (n-major rows) in shared memory:
//   dh_{t-1} = z * dh + W_hh^T [dr_pre, dz_pre, r * dn_pre]; it writes the gradient of the input
//   projection (dgx) and the hidden-side n-gate gradient; the weight gradients are GEMMs over
//   those arrays on the host side.
#include "isa_common.cuh"
#include "isa_ptx.cuh"
#include "isa_tcgen05.cuh"
#include <math.h>

namespace {

struct TokMap {
  int inner;
  long long outer_stride, inner_stride, t_stride;  // in tokens
};
__device__ __forceinline__ long long tok_base(const TokMap& m, int q) {
  return (long long)(q / m.inner) * m.outer_stride + (long long)(q % m.inner) * m.inner_stride;
}

__device__ __forceinline__ float sigmoidf_acc(float x) { return 1.f / (1.f + expf(-x)); }

struct GruFwdParams {
  const float* gx;     // [tokens][2][3n]
  const float* w_hh;   // [2][3n][n]
  const float* b_hh;   // [2][3n]
  const float* b_ih;   // [2][3n] or null: input-side bias when gx = x W_ih^T carries none
  float* out;          // [tokens][2n]
  float* stash;        // [tokens][2][4n] (r, z, n, hn) or null
  int n_seq, T, n;
  TokMap map;
};

// S sequences per CTA, ST = S/2 per thread; thread = (unit j, sequence half sg)
template <int S>
__global__ void __launch_bounds__(256, 1) gru_scan_fwd_kernel(const GruFwdParams prm) {
  constexpr int ST = S / 2;
  extern __shared__ __align__(16) float smem[];
  const int n = prm.n, n3 = 3 * n;
  float* s_wt = smem;                   // [n][3n]   W_hh^T
  float* s_h = s_wt + (size_t)n * n3;   // [2][n][S]
  const int d = blockIdx.y;
  const int q0 = blockIdx.x * S;
  const int T = prm.T;

  // W_hh^T -> smem (one-time; coalesced global reads along i)
  const float* __restrict__ w = prm.w_hh + (size_t)d * n3 * n;
  for (int idx = threadIdx.x; idx < n3 * n; idx += blockDim.x) {
    const int g = idx / n, i = idx % n;
    s_wt[(size_t)i * n3 + g] = __ldg(w + idx);
  }
  for (int idx = threadIdx.x; idx < 2 * n * S; idx += blockDim.x) s_h[idx] = 0.f;

  const int j = threadIdx.x % n;     // hidden unit (threads >= 2n idle in the math)
  const int sg = threadIdx.x / n;    // 0 or 1
  const bool active = threadIdx.x < 2 * n;
  const float bhr = active ? __ldg(prm.b_hh + d * n3 + j) + (prm.b_ih ? __ldg(prm.b_ih + d * n3 + j) : 0.f) : 0.f;
  const float bhz = active ? __ldg(prm.b_hh + d * n3 + n + j) + (prm.b_ih ? __ldg(prm.b_ih + d * n3 + n + j) : 0.f) : 0.f;
  const float bhn = active ? __ldg(prm.b_hh + d * n3 + 2 * n + j) : 0.f;
  const float bin = (active && prm.b_ih) ? __ldg(prm.b_ih + d * n3 + 2 * n + j) : 0.f;

  long long base[ST];
  bool valid[ST];
#pragma unroll
  for (int s = 0; s < ST; ++s) {
    const int q = q0 + sg * ST + s;
    valid[s] = active && q < prm.n_seq;
    base[s] = valid[s] ? tok_base(prm.map, q) : 0;
  }
  const float* __restrict__ gx = prm.gx + (size_t)d * n3 + j;

  float gr[ST], gz[ST], gn[ST];  // prefetched x-projection of the coming step
  auto prefetch = [&](int t) {
#pragma unroll
    for (int s = 0; s < ST; ++s) {
      if (valid[s]) {
        const float* p = gx + (size_t)(base[s] + (long long)t * prm.map.t_stride) * (2 * n3);
        gr[s] = __ldg(p); gz[s] = __ldg(p + n); gn[s] = __ldg(p + 2 * n);
      } else { gr[s] = gz[s] = gn[s] = 0.f; }
    }
  };
  prefetch(d == 0 ? 0 : T - 1);
  __syncthreads();

  for (int step = 0; step < T; ++step) {
    const int t = (d == 0) ? step : T - 1 - step;
    const float* __restrict__ hc = s_h + (size_t)(step & 1) * n * S;
    float* __restrict__ hn_buf = s_h + (size_t)((step + 1) & 1) * n * S;
    float xr[ST], xz[ST], xn[ST];
#pragma unroll
    for (int s = 0; s < ST; ++s) { xr[s] = gr[s]; xz[s] = gz[s]; xn[s] = gn[s]; }
    if (step + 1 < T) prefetch(d == 0 ? step + 1 : T - 2 - step);

    if (active) {
      float ar[ST], az[ST], an[ST];
#pragma unroll
      for (int s = 0; s < ST; ++s) { ar[s] = 0.f; az[s] = 0.f; an[s] = 0.f; }
      const float* __restrict__ wp = s_wt + j;
      const float* __restrict__ hp = hc + sg * ST;
#pragma unroll 4
      for (int i = 0; i < n; ++i) {
        const float wr = wp[(size_t)i * n3], wz = wp[(size_t)i * n3 + n], wn = wp[(size_t)i * n3 + 2 * n];
        float hv[ST];
#pragma unroll
        for (int s4 = 0; s4 < ST; s4 += 4) {
          if (ST >= 4) {
            const float4 v = *reinterpret_cast<const float4*>(hp + (size_t)i * S + s4);
            hv[s4] = v.x; hv[s4 + 1] = v.y; hv[s4 + 2] = v.z; hv[s4 + 3] = v.w;
          }
        }
        if (ST < 4) {
#pragma unroll
          for (int s = 0; s < ST; ++s) hv[s] = hp[(size_t)i * S + s];
        }
#pragma unroll
        for (int s = 0; s < ST; ++s) {
          ar[s] = fmaf(wr, hv[s], ar[s]);
          az[s] = fmaf(wz, hv[s], az[s]);
          an[s] = fmaf(wn, hv[s], an[s]);
        }
      }
#pragma unroll
      for (int s = 0; s < ST; ++s) {
        const float hprev = hc[(size_t)j * S + sg * ST + s];
        const float r = sigmoidf_acc(xr[s] + ar[s] + bhr);
        const float z = sigmoidf_acc(xz[s] + az[s] + bhz);
        const float hnn = an[s] + bhn;
        const float nn = tanhf(xn[s] + bin + r * hnn);
        const float hnew = (1.f - z) * nn + z * hprev;
        hn_buf[(size_t)j * S + sg * ST + s] = hnew;
        if (valid[s]) {
          const long long tok = base[s] + (long long)t * prm.map.t_stride;
          prm.out[(size_t)tok * (2 * n) + d * n + j] = hnew;
          if (prm.stash) {
            float* st = prm.stash + ((size_t)tok * 2 + d) * (4 * n) + j;
            st[0] = r; st[n] = z; st[2 * n] = nn; st[3 * n] = hnn;
          }
        }
      }
    }
    __syncthreads();
  }
}

struct GruBwdParams {
  const float* dout;   // [tokens][2n]
  const float* out;    // [tokens][2n]  forward output (h_t)
  const float* stash;  // [tokens][2][4n]
  const float* w_hh;   // [2][3n][n]
  float* dgx;          // [tokens][2][3n]
  float* dghn;         // [tokens][2][n]   r * dn_pre (hidden-side n-gate gradient)
  int n_seq, T, n;
  TokMap map;
};

template <int S>
__global__ void __launch_bounds__(256, 1) gru_scan_bwd_kernel(const GruBwdParams prm) {
  constexpr int ST = S / 2;
  extern __shared__ __align__(16) float smem[];
  const int n = prm.n, n3 = 3 * n;
  float* s_w = smem;                     // [3n][n]  W_hh as stored
  float* s_dg = s_w + (size_t)n3 * n;    // [3n][S]  hidden-side gate gradients of this step
  float* s_dh = s_dg + (size_t)n3 * S;   // [n][S]   dh carried to the previous step
  const int d = blockIdx.y;
  const int q0 = blockIdx.x * S;
  const int T = prm.T;
  const float* __restrict__ w = prm.w_hh + (size_t)d * n3 * n;
  for (int idx = threadIdx.x; idx < n3 * n; idx += blockDim.x) s_w[idx] = __ldg(w + idx);
  for (int idx = threadIdx.x; idx < n * S; idx += blockDim.x) s_dh[idx] = 0.f;

  const int j = threadIdx.x % n;
  const int sg = threadIdx.x / n;
  const bool active = threadIdx.x < 2 * n;
  long long base[ST];
  bool valid[ST];
#pragma unroll
  for (int s = 0; s < ST; ++s) {
    const int q = q0 + sg * ST + s;
    valid[s] = active && q < prm.n_seq;
    base[s] = valid[s] ? tok_base(prm.map, q) : 0;
  }
  __syncthreads();

  // backward visits the steps in the opposite order of the forward sweep of this direction
  for (int step = T - 1; step >= 0; --step) {
    const int t = (d == 0) ? step : T - 1 - step;        // token position of forward step `step`
    const int tp = (d == 0) ? t - 1 : t + 1;             // position holding h_{step-1}
    if (active) {
#pragma unroll
      for (int s = 0; s < ST; ++s) {
        float dr_pre = 0.f, dz_pre = 0.f, dn_pre = 0.f, dnr = 0.f, dh_direct = 0.f;
        if (valid[s]) {
          const long long tok = base[s] + (long long)t * prm.map.t_stride;
          const float* st = prm.stash + ((size_t)tok * 2 + d) * (4 * n) + j;
          const float r = __ldg(st), z = __ldg(st + n), nn = __ldg(st + 2 * n), hnn = __ldg(st + 3 * n);
          float hprev = 0.f;
          if (step > 0) hprev = __ldg(prm.out + (size_t)(base[s] + (long long)tp * prm.map.t_stride) * (2 * n) + d * n + j);
          const float dh = __ldg(prm.dout + (size_t)tok * (2 * n) + d * n + j) + s_dh[(size_t)j * S + sg * ST + s];
          const float dn = dh * (1.f - z);
          const float dz = dh * (hprev - nn);
          dh_direct = dh * z;
          dn_pre = dn * (1.f - nn * nn);
          dz_pre = dz * z * (1.f - z);
          dr_pre = dn_pre * hnn * r * (1.f - r);
          dnr = dn_pre * r;
          float* g = prm.dgx + ((size_t)tok * 2 + d) * n3 + j;
          g[0] = dr_pre; g[n] = dz_pre; g[2 * n] = dn_pre;
          prm.dghn[((size_t)tok * 2 + d) * n + j] = dnr;
        }
        s_dg[(size_t)j * S + sg * ST + s] = dr_pre;
        s_dg[(size_t)(n + j) * S + sg * ST + s] = dz_pre;
        s_dg[(size_t)(2 * n + j) * S + sg * ST + s] = dnr;
        // stash the direct term in registers via smem slot reuse below
        s_dh[(size_t)j * S + sg * ST + s] = dh_direct;
      }
    }
    __syncthreads();
    if (active) {
      // dh_{step-1}[i=j] = z*dh + sum_g W_hh[g][j] * dg[g]
      float acc[ST];
#pragma unroll
      for (int s = 0; s < ST; ++s) acc[s] = 0.f;
      const float* __restrict__ wp = s_w + j;
      const float* __restrict__ gp = s_dg + sg * ST;
#pragma unroll 4
      for (int g = 0; g < n3; ++g) {
        const float wv = wp[(size_t)g * n];
        float gv[ST];
#pragma unroll
        for (int s4 = 0; s4 < ST; s4 += 4) {
          if (ST >= 4) {
            const float4 v = *reinterpret_cast<const float4*>(gp + (size_t)g * S + s4);
            gv[s4] = v.x; gv[s4 + 1] = v.y; gv[s4 + 2] = v.z; gv[s4 + 3] = v.w;
          }
        }
        if (ST < 4) {
#pragma unroll
          for (int s = 0; s < ST; ++s) gv[s] = gp[(size_t)g * S + s];
        }
#pragma unroll
        for (int s = 0; s < ST; ++s) acc[s] = fmaf(wv, gv[s], acc[s]);
      }
#pragma unroll
      for (int s = 0; s < ST; ++s) s_dh[(size_t)j * S + sg * ST + s] += acc[s];
    }
    __syncthreads();
  }
}

// ================================================================================================ tensor-core scan
// The recurrent product of a step, G[3n x S] = W_hh[3n x n] h[n x S], on the 5th-generation tensor cores:
//   * W_hh lives in TENSOR MEMORY for the whole sweep as the A operand (one 128-row tile per gate, rows = hidden
//     units, bf16 hi and lo parts: 6 x 56 = 336 columns for n = 100), so a step's MMAs read only the 7 KB B operand;
//   * h_{t-1} of the CTA's <= 16 sequences is the B operand [N = 16][K = n] in shared memory (bf16 hi / lo, canonical
//     K-major core matrices), rewritten every step by the gate threads;
//   * every product is a_hi b_hi + a_hi b_lo + a_lo b_hi with fp32 accumulation (error ~2^-16, like the projections):
//     3 gates x 7 k-steps x 3 = 63 tcgen05.mma (N = 16) per step, ~0.5 k cycles, issued warp-uniformly by one warp;
//   * the accumulators D_g [128 x 16] come back with tcgen05.ld: TMEM lane = hidden unit, so thread j holds the three
//     gate pre-activations of unit j for all 16 sequences and does the gate math (ex2 / rcp on the MUFU), keeps h in
//     registers, stores h / the stash rows (coalesced over j) and writes the next B operand;
//   * the per-step gx rows arrive through a 3-stage TMA bulk-copy ring filled by a dedicated producer warp.
// A step is ~1.5 k cycles of latency (MMA 0.5 k + gate math 0.7 k + hand-offs), below the ~2.3 k cycles the step's HBM
// traffic costs at 148 CTAs.  Keeping W_hh in registers with FFMA2 inner products instead was measured at 8.6 k cycles
// per step (DESIGN.md).
template <int NU>
struct TcCfg {
  static constexpr int KP = (NU + 15) / 16 * 16;      // reduction length padded to the MMA's K = 16
  static constexpr int KSTEPS = KP / 16;
  static constexpr int ACOLS = KP / 2;                // TMEM columns of one (gate, part) A tile: packed bf16 pairs
  static constexpr int TM_D = 6 * ACOLS;              // accumulators: chain c, gate g at TM_D + 48 c + 16 g
  static constexpr int NSEQ = 16;                     // MMA N
  static constexpr int SBO_B = (KP / 8) * 128;        // byte stride between 8-sequence groups of the B operand
  static constexpr int B_PART = 2 * SBO_B;            // bytes of one part (hi or lo) of B
  static constexpr int STAGES = 5;
  // Two independent chains of 8 sequences each (every MMA still spans all N = 16 columns; a chain reads back only its
  // own columns of its own accumulators): while one chain's MMAs and hand-offs are in flight the other chain's gate
  // threads compute, so neither the gate math nor the tensor pipe waits for the other.
  static constexpr int NT = 640;                      // warp 0 producer, warps 1-2 MMA issuers, warp 3 idle, warps 4..19 gate threads
  static constexpr int CHAIN_THREADS = 256;           // per chain: (TMEM quarter = warp % 4) x (4-sequence half)
  static constexpr size_t gx_bytes = (size_t)STAGES * NSEQ * 3 * NU * sizeof(float);
  static constexpr size_t used_bytes = gx_bytes + 2 * B_PART + 16 * 8 + NSEQ * 8 + 16 + 128;
  // the CTA allocates all 512 TMEM columns: ask for more than half of the SM's shared memory so that two CTAs can never
  // share an SM (the second one would spin in tcgen05.alloc until the first retires)
  static constexpr size_t smem_bytes = used_bytes > 120 * 1024 ? used_bytes : 120 * 1024;
  static_assert(TM_D + 2 * 3 * 16 <= 512 && NU <= 128 && NU % 4 == 0, "unsupported width");
};

__device__ __forceinline__ float sigmoid_fast(float x) { return __fdividef(1.f, 1.f + ex2_approx(-1.4426950408889634f * x)); }
__device__ __forceinline__ float tanh_fast(float x) { return fmaf(2.f, __fdividef(1.f, 1.f + ex2_approx(-2.8853900817779268f * x)), -1.f); }

template <int NU>
__global__ void __launch_bounds__(TcCfg<NU>::NT, 1) gru_fwd_tc_kernel(const GruFwdParams prm, const int S) {
  using Cfg = TcCfg<NU>;
  constexpr int N3 = 3 * NU, NSEQ = Cfg::NSEQ, STAGES = Cfg::STAGES;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  unsigned char* sm = smem_raw + ((128u - (smem_u32(smem_raw) & 127u)) & 127u);
  float* s_gx = reinterpret_cast<float*>(sm);                               // [STAGES][16][3n]
  unsigned char* s_b = sm + Cfg::gx_bytes;                                   // B operand: hi part | lo part
  uint64_t* s_bar = reinterpret_cast<uint64_t*>(s_b + 2 * Cfg::B_PART);      // gx_full[3] gx_empty[3] h_full d_full
  long long* s_tok = reinterpret_cast<long long*>(s_bar + 16);
  uint32_t* s_tmem = reinterpret_cast<uint32_t*>(s_tok + NSEQ);
  uint64_t* gx_full = s_bar;
  uint64_t* gx_empty = s_bar + STAGES;
  uint64_t* h_full = s_bar + 2 * STAGES;          // [2] per chain
  uint64_t* d_full = s_bar + 2 * STAGES + 2;      // [2]

  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;
  const int d = blockIdx.y;
  const int q0 = blockIdx.x * S;
  const int T = prm.T;
  const int n_valid = min(S, prm.n_seq - q0);

  if (threadIdx.x == 0) {
    for (int i = 0; i < STAGES; ++i) { mbar_init(&gx_full[i], 1); mbar_init(&gx_empty[i], 2 * Cfg::CHAIN_THREADS); }
    for (int c = 0; c < 2; ++c) { mbar_init(&h_full[c], Cfg::CHAIN_THREADS); mbar_init(&d_full[c], 1); }
    fence_barrier_init();
  }
  for (int i = threadIdx.x; i < (int)((Cfg::gx_bytes + 2 * Cfg::B_PART) / 4); i += Cfg::NT) reinterpret_cast<uint32_t*>(sm)[i] = 0u;
  if (threadIdx.x < NSEQ) s_tok[threadIdx.x] = (int)threadIdx.x < n_valid ? tok_base(prm.map, q0 + threadIdx.x) : -1;
  if (warp == 1) tmem_alloc(s_tmem, 512);
  fence_proxy_async();          // the zero-filled B operand is read through the async proxy by the first MMAs
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *s_tmem;

  const int quarter = warp & 3;
  const int j = quarter * 32 + lane;                       // hidden unit of a gate thread = TMEM lane
  const uint32_t t_row = tmem + ((uint32_t)(quarter * 32) << 16);
  if (warp >= 4) {
    // W_hh -> TMEM (once): row j of gate g, split into bf16 hi / lo, two values per 32-bit column; the (gate, k-chunk)
    // items are dealt round-robin to the four warps that share a TMEM quarter
    const float* __restrict__ wsrc = prm.w_hh + (size_t)d * N3 * NU;
#pragma unroll 1
    for (int item = (warp - 4) >> 2; item < 3 * Cfg::KSTEPS; item += 4) {
      const int g = item / Cfg::KSTEPS, c = item % Cfg::KSTEPS;
      {
        uint32_t hi[8], lo[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) {
          const int k = c * 16 + 2 * e;
          float a = 0.f, b = 0.f;
          if (j < NU && k < NU) {          // NU even: k and k + 1 are valid together
            // two scalar loads: the C-ABI promises w_hh only fp32 alignment, so a float2 load could be misaligned
            const float* p = wsrc + (size_t)(g * NU + j) * NU + k;
            a = __ldg(p); b = __ldg(p + 1);
          }
          split2(a, b, hi[e], lo[e]);
        }
        tmem_st8_issue(t_row + (g * 2) * Cfg::ACOLS + c * 8, hi);
        tmem_st8_issue(t_row + (g * 2 + 1) * Cfg::ACOLS + c * 8, lo);
      }
    }
    tmem_st_wait();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();

  if (warp == 0) {
    // ===================== producer: gx rows of step st -> stage st % STAGES =====================
    for (int st = 0; st < T; ++st) {
      const int stage = st % STAGES;
      mbar_wait(&gx_empty[stage], ((st / STAGES) & 1) ^ 1);
      if (lane == 0) mbar_arrive_expect_tx(&gx_full[stage], (uint32_t)n_valid * N3 * 4u);
      __syncwarp();
      if (lane < n_valid) {
        const int t = (d == 0) ? st : T - 1 - st;
        const long long tok = s_tok[lane] + (long long)t * prm.map.t_stride;
        tma_bulk_g2s(s_gx + ((size_t)stage * NSEQ + lane) * N3, prm.gx + ((size_t)tok * 2 + d) * N3, N3 * 4u, &gx_full[stage]);
      }
    }
  } else if (warp <= 2) {
    // ===================== MMA issuer of chain c = warp - 1 (warp-uniform, one elected lane) =====================
    const int c = warp - 1;
    const uint32_t el = elect_one();
    constexpr uint32_t idesc = make_idesc(128, NSEQ);
    const uint64_t b_hi = make_desc(smem_u32(s_b), 128, Cfg::SBO_B);
    const uint64_t b_lo = make_desc(smem_u32(s_b + Cfg::B_PART), 128, Cfg::SBO_B);
    for (int step = 0; step < T; ++step) {
      if (step > 0) mbar_wait(&h_full[c], (step - 1) & 1);
      tc_fence_after();
      // consecutive MMAs go to different accumulators (gates): back-to-back accumulations into the SAME TMEM tile would
      // serialise on the tensor pipe's latency, far above the 8 cycles an N = 16 MMA occupies it
#pragma unroll
      for (int kk = 0; kk < Cfg::KSTEPS; ++kk) {
        const uint32_t ko = (kk * 256) >> 4;
#pragma unroll
        for (int term = 0; term < 3; ++term) {
#pragma unroll
          for (int g = 0; g < 3; ++g) {
            const uint32_t dcol = tmem + Cfg::TM_D + c * 48 + g * 16;
            const uint32_t a = tmem + (g * 2 + (term == 2 ? 1 : 0)) * Cfg::ACOLS + kk * 8;
            umma_bf16_ts_e(el, dcol, a, (term == 1 ? b_lo : b_hi) + ko, idesc, (kk > 0 || term > 0) ? 1u : 0u);
          }
        }
      }
      umma_commit_e(el, &d_full[c]);
    }
  } else if (warp >= 4) {
    // ===================== gate threads: unit j, four sequences of chain c =====================
    constexpr int SH = 4;
    const int sub = (warp - 4) >> 2;                       // 0..3
    const int c = sub >> 1;
    const int s0 = c * 8 + (sub & 1) * SH;                 // first sequence of this thread
    const bool unit = j < NU;
    const int jj = unit ? j : 0;
    const float bhr = __ldg(prm.b_hh + d * N3 + jj) + (prm.b_ih ? __ldg(prm.b_ih + d * N3 + jj) : 0.f);
    const float bhz = __ldg(prm.b_hh + d * N3 + NU + jj) + (prm.b_ih ? __ldg(prm.b_ih + d * N3 + NU + jj) : 0.f);
    const float bhn = __ldg(prm.b_hh + d * N3 + 2 * NU + jj);
    const float bin = prm.b_ih ? __ldg(prm.b_ih + d * N3 + 2 * NU + jj) : 0.f;
    float hreg[SH];
    // running output pointers: one 64-bit add per sequence and step instead of the token arithmetic
    float* po[SH];
    float* ps[SH];
    uint32_t valid = 0;
    const long long t_first = (d == 0) ? 0 : T - 1;
    const long long dstep = ((d == 0) ? 1 : -1) * prm.map.t_stride;
#pragma unroll
    for (int s = 0; s < SH; ++s) {
      hreg[s] = 0.f;
      const long long tb = s_tok[s0 + s];
      const long long tok = (tb >= 0 ? tb : 0) + t_first * prm.map.t_stride;
      if (tb >= 0) valid |= 1u << s;
      po[s] = prm.out + (size_t)tok * (2 * NU) + d * NU + jj;
      ps[s] = prm.stash ? prm.stash + ((size_t)tok * 2 + d) * (4 * NU) + jj : nullptr;
    }
    const long long dout = dstep * (2 * NU), dstash = dstep * (8 * NU);
    const bool has_stash = prm.stash != nullptr;
    // sequence s0 + s: row group (s0 + s) / 8 = c, row (s0 + s) % 8 inside the core matrices
    unsigned char* b_base = s_b + (jj >> 3) * 128 + (jj & 7) * 2 + c * Cfg::SBO_B + (s0 & 7) * 16;
    const uint32_t t_d = t_row + Cfg::TM_D + c * 48 + s0;
    for (int step = 0; step < T; ++step) {
      const int stage = step % STAGES;
      mbar_wait(&d_full[c], step & 1);
      tc_fence_after();
      uint32_t ar[SH], az[SH], an[SH];
      tmem_ld4_issue(t_d, ar);
      tmem_ld4_issue(t_d + 16, az);
      tmem_ld4_issue(t_d + 32, an);
      tmem_ld4_wait(ar);
      tmem_ld4_wait(az);
      tmem_ld4_wait(an);
      mbar_wait(&gx_full[stage], (step / STAGES) & 1);
      const float* __restrict__ gxs = s_gx + ((size_t)stage * NSEQ + s0) * N3 + jj;
      float hn[SH], r[SH], z[SH], nn[SH];
      if (unit) {
        // staged over the thread's sequences so that the four dependent MUFU chains run interleaved, not one after another
        constexpr float kL2E = 1.4426950408889634f;
        float pr[SH], pz[SH], pn[SH];
#pragma unroll
        for (int s = 0; s < SH; ++s) {
          pr[s] = gxs[s * N3] + __uint_as_float(ar[s]) + bhr;
          pz[s] = gxs[s * N3 + NU] + __uint_as_float(az[s]) + bhz;
          pn[s] = gxs[s * N3 + 2 * NU] + bin;
          hn[s] = __uint_as_float(an[s]) + bhn;
        }
#pragma unroll
        for (int s = 0; s < SH; ++s) { pr[s] = ex2_approx(-kL2E * pr[s]); pz[s] = ex2_approx(-kL2E * pz[s]); }
#pragma unroll
        for (int s = 0; s < SH; ++s) { r[s] = __fdividef(1.f, 1.f + pr[s]); z[s] = __fdividef(1.f, 1.f + pz[s]); }
#pragma unroll
        for (int s = 0; s < SH; ++s) pn[s] = ex2_approx(-2.f * kL2E * fmaf(r[s], hn[s], pn[s]));
#pragma unroll
        for (int s = 0; s < SH; ++s) nn[s] = fmaf(2.f, __fdividef(1.f, 1.f + pn[s]), -1.f);
#pragma unroll
        for (int s = 0; s < SH; ++s) hreg[s] = fmaf(z[s], hreg[s] - nn[s], nn[s]);        // (1 - z) n + z h
#pragma unroll
        for (int s = 0; s < SH; ++s) {
          const __nv_bfloat16 hh = __float2bfloat16_rn(hreg[s]);
          const __nv_bfloat16 hl = __float2bfloat16_rn(hreg[s] - __bfloat162float(hh));
          unsigned char* bp = b_base + s * 16;
          *reinterpret_cast<__nv_bfloat16*>(bp) = hh;
          *reinterpret_cast<__nv_bfloat16*>(bp + Cfg::B_PART) = hl;
        }
      }
      tc_fence_before();
      fence_proxy_async();          // B operand writes -> visible to the tensor core's async proxy
      mbar_arrive(&h_full[c]);
      mbar_arrive(&gx_empty[stage]);
      // global stores AFTER the hand-off: mbarrier.arrive has release semantics, so stores issued before it would have
      // to be acknowledged (~1 k cycles) before the next step's MMAs could start; here they drain under the MMAs
      if (unit) {
#pragma unroll
        for (int s = 0; s < SH; ++s) {
          if ((valid >> s) & 1u) {
            *po[s] = hreg[s];
            if (has_stash) {
              float* st4 = ps[s];
              st4[0] = r[s]; st4[NU] = z[s]; st4[2 * NU] = nn[s]; st4[3 * NU] = hn[s];
            }
          }
          po[s] += dout;
          ps[s] += dstash;
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem, 512);
}

template <int NU>
int launch_fwd_tc(const GruFwdParams& prm, int S, cudaStream_t stream) {
  using Cfg = TcCfg<NU>;
  ISA_CUDA(cudaFuncSetAttribute(gru_fwd_tc_kernel<NU>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Cfg::smem_bytes));
  dim3 grid((prm.n_seq + S - 1) / S, 2);
  gru_fwd_tc_kernel<NU><<<grid, Cfg::NT, Cfg::smem_bytes, stream>>>(prm, S);
  return ISA_OK;
}


// ---- backward (BPTT) on the tensor cores: dh_{t-1}[u] = z dh[u] + sum_g W_hh[g][u] dg[g], with W_hh^T [n x 3n] resident
// in TMEM as the A operand (2 x 152 columns for n = 100), the step's gate gradients dg = (dr_pre, dz_pre, r dn_pre) of the
// <= 16 sequences as the B operand [16][3n] in shared memory (bf16 hi / lo), 19 k-steps x 3 = 57 MMAs per step.
// Gate threads: unit j x eight sequences; their inputs (stash row, h_{t-1}, dL/dh_t) arrive through a TMA ring.
template <int NU>
struct TcBwdCfg {
  static constexpr int K3 = 3 * NU;
  static constexpr int KP = (K3 + 15) / 16 * 16;
  static constexpr int KSTEPS = KP / 16;
  static constexpr int ACOLS = KP / 2;
  static constexpr int TM_D = 2 * ACOLS;
  static constexpr int NSEQ = 16;
  static constexpr int SBO_B = (KP / 8) * 128;
  static constexpr int B_PART = 2 * SBO_B;
  static constexpr int STAGES = 4;
  static constexpr int ROW = 6 * NU;                  // floats per sequence and stage: stash 4n | h_prev n | dout n
  static constexpr int NT = 640;                      // same roles and two-chain organisation as the forward kernel
  static constexpr int CHAIN_THREADS = 256;
  static constexpr size_t in_bytes = (size_t)STAGES * NSEQ * ROW * sizeof(float);
  static constexpr size_t used_bytes = in_bytes + 2 * B_PART + 16 * 8 + NSEQ * 8 + 16 + 128;
  static constexpr size_t smem_bytes = used_bytes > 120 * 1024 ? used_bytes : 120 * 1024;
  static_assert(TM_D + 2 * 16 <= 512 && NU <= 128 && NU % 4 == 0, "unsupported width");
};

template <int NU>
__global__ void __launch_bounds__(TcBwdCfg<NU>::NT, 1) gru_bwd_tc_kernel(const GruBwdParams prm, const int S) {
  using Cfg = TcBwdCfg<NU>;
  constexpr int N3 = 3 * NU, NSEQ = Cfg::NSEQ, STAGES = Cfg::STAGES, ROW = Cfg::ROW;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  unsigned char* sm = smem_raw + ((128u - (smem_u32(smem_raw) & 127u)) & 127u);
  float* s_in = reinterpret_cast<float*>(sm);                                // [STAGES][16][ROW]
  unsigned char* s_b = sm + Cfg::in_bytes;                                   // B operand: hi part | lo part
  uint64_t* s_bar = reinterpret_cast<uint64_t*>(s_b + 2 * Cfg::B_PART);
  long long* s_tok = reinterpret_cast<long long*>(s_bar + 16);
  uint32_t* s_tmem = reinterpret_cast<uint32_t*>(s_tok + NSEQ);
  uint64_t* in_full = s_bar;
  uint64_t* in_empty = s_bar + STAGES;
  uint64_t* g_full = s_bar + 2 * STAGES;          // [2] per chain
  uint64_t* d_full = s_bar + 2 * STAGES + 2;      // [2]

  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;
  const int d = blockIdx.y;
  const int q0 = blockIdx.x * S;
  const int T = prm.T;
  const int n_valid = min(S, prm.n_seq - q0);

  if (threadIdx.x == 0) {
    for (int i = 0; i < STAGES; ++i) { mbar_init(&in_full[i], 1); mbar_init(&in_empty[i], 2 * Cfg::CHAIN_THREADS); }
    for (int c = 0; c < 2; ++c) { mbar_init(&g_full[c], Cfg::CHAIN_THREADS); mbar_init(&d_full[c], 1); }
    fence_barrier_init();
  }
  for (int i = threadIdx.x; i < (int)((Cfg::in_bytes + 2 * Cfg::B_PART) / 4); i += Cfg::NT) reinterpret_cast<uint32_t*>(sm)[i] = 0u;
  if (threadIdx.x < NSEQ) s_tok[threadIdx.x] = (int)threadIdx.x < n_valid ? tok_base(prm.map, q0 + threadIdx.x) : -1;
  if (warp == 1) tmem_alloc(s_tmem, 512);
  fence_proxy_async();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *s_tmem;

  const int quarter = warp & 3;
  const int j = quarter * 32 + lane;
  const uint32_t t_row = tmem + ((uint32_t)(quarter * 32) << 16);
  if (warp >= 4) {
    // W_hh^T -> TMEM (once): row u = j holds W_hh[g][u] over g, bf16 hi / lo pairs (coalesced: lanes run along u); the
    // k-chunks are dealt round-robin to the four warps that share a TMEM quarter
    const float* __restrict__ wsrc = prm.w_hh + (size_t)d * N3 * NU;
#pragma unroll 1
    for (int c = (warp - 4) >> 2; c < Cfg::KSTEPS; c += 4) {
      uint32_t hi[8], lo[8];
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        const int g = c * 16 + 2 * e;
        const float a = (j < NU && g < N3) ? __ldg(wsrc + (size_t)g * NU + j) : 0.f;
        const float b = (j < NU && g + 1 < N3) ? __ldg(wsrc + (size_t)(g + 1) * NU + j) : 0.f;
        split2(a, b, hi[e], lo[e]);
      }
      tmem_st8_issue(t_row + c * 8, hi);
      tmem_st8_issue(t_row + Cfg::ACOLS + c * 8, lo);
    }
    tmem_st_wait();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();

  if (warp == 0) {
    // ===================== producer: rows of forward step T-1-it -> stage it % STAGES =====================
    for (int it = 0; it < T; ++it) {
      const int st = T - 1 - it;
      const int stage = it % STAGES;
      mbar_wait(&in_empty[stage], ((it / STAGES) & 1) ^ 1);
      const uint32_t per_seq = (st > 0 ? 6u : 5u) * NU * 4u;
      if (lane == 0) mbar_arrive_expect_tx(&in_full[stage], (uint32_t)n_valid * per_seq);
      __syncwarp();
      if (lane < n_valid) {
        const int t = (d == 0) ? st : T - 1 - st;
        const int tp = (d == 0) ? t - 1 : t + 1;
        const long long b0 = s_tok[lane];
        const long long tok = b0 + (long long)t * prm.map.t_stride;
        float* dst = s_in + ((size_t)stage * NSEQ + lane) * ROW;
        tma_bulk_g2s(dst, prm.stash + ((size_t)tok * 2 + d) * (4 * NU), 4u * NU * 4u, &in_full[stage]);
        if (st > 0) {
          const long long tokp = b0 + (long long)tp * prm.map.t_stride;
          tma_bulk_g2s(dst + 4 * NU, prm.out + (size_t)tokp * (2 * NU) + d * NU, NU * 4u, &in_full[stage]);
        }
        tma_bulk_g2s(dst + 5 * NU, prm.dout + (size_t)tok * (2 * NU) + d * NU, NU * 4u, &in_full[stage]);
      }
    }
  } else if (warp <= 2) {
    // ===================== MMA issuer of chain c = warp - 1 =====================
    const int c = warp - 1;
    const uint32_t el = elect_one();
    constexpr uint32_t idesc = make_idesc(128, NSEQ);
    const uint64_t b_hi = make_desc(smem_u32(s_b), 128, Cfg::SBO_B);
    const uint64_t b_lo = make_desc(smem_u32(s_b + Cfg::B_PART), 128, Cfg::SBO_B);
    const uint32_t dcol = tmem + Cfg::TM_D + c * 16;
    for (int it = 0; it + 1 < T; ++it) {                 // the last step's dh_{-1} is not needed
      mbar_wait(&g_full[c], it & 1);
      tc_fence_after();
#pragma unroll
      for (int kk = 0; kk < Cfg::KSTEPS; ++kk) {
        const uint32_t a_hi = tmem + kk * 8, a_lo = tmem + Cfg::ACOLS + kk * 8;
        const uint32_t ko = (kk * 256) >> 4;
        umma_bf16_ts_e(el, dcol, a_hi, b_hi + ko, idesc, kk > 0 ? 1u : 0u);
        umma_bf16_ts_e(el, dcol, a_hi, b_lo + ko, idesc, 1u);
        umma_bf16_ts_e(el, dcol, a_lo, b_hi + ko, idesc, 1u);
      }
      umma_commit_e(el, &d_full[c]);
    }
  } else if (warp >= 4) {
    // ===================== gate threads: unit j, four sequences of chain c =====================
    constexpr int SH = 4;
    const int sub = (warp - 4) >> 2;
    const int c = sub >> 1;
    const int s0 = c * 8 + (sub & 1) * SH;
    const bool unit = j < NU;
    const int jj = unit ? j : 0;
    float dhd[SH];
    float* pg[SH];
    float* pn[SH];
    uint32_t valid = 0;
    const long long t_first = (d == 0) ? T - 1 : 0;       // time index of forward step T-1
    const long long dstep = ((d == 0) ? -1 : 1) * prm.map.t_stride;
#pragma unroll
    for (int s = 0; s < SH; ++s) {
      dhd[s] = 0.f;
      const long long tb = s_tok[s0 + s];
      const long long tok = (tb >= 0 ? tb : 0) + t_first * prm.map.t_stride;
      if (tb >= 0) valid |= 1u << s;
      pg[s] = prm.dgx + ((size_t)tok * 2 + d) * N3 + jj;
      pn[s] = prm.dghn + ((size_t)tok * 2 + d) * NU + jj;
    }
    const long long dg_stride = dstep * (2 * N3), dn_stride = dstep * (2 * NU);
    // B operand slots of this unit's three gate rows k = j, n + j, 2n + j
    unsigned char* b_seq = s_b + c * Cfg::SBO_B + (s0 & 7) * 16;
    const int k1 = NU + jj, k2 = 2 * NU + jj;
    const int o0 = (jj >> 3) * 128 + (jj & 7) * 2, o1 = (k1 >> 3) * 128 + (k1 & 7) * 2, o2 = (k2 >> 3) * 128 + (k2 & 7) * 2;
    const uint32_t t_d = t_row + Cfg::TM_D + c * 16 + s0;
    for (int it = 0; it < T; ++it) {
      const int step = T - 1 - it;
      const int stage = it % STAGES;
      mbar_wait(&in_full[stage], (it / STAGES) & 1);
      float dprev[SH];
      if (it > 0) {
        mbar_wait(&d_full[c], (it - 1) & 1);
        tc_fence_after();
        uint32_t dr[SH];
        tmem_ld4_issue(t_d, dr);
        tmem_ld4_wait(dr);
#pragma unroll
        for (int s = 0; s < SH; ++s) dprev[s] = dhd[s] + __uint_as_float(dr[s]);
      } else {
#pragma unroll
        for (int s = 0; s < SH; ++s) dprev[s] = 0.f;
      }
      const float* __restrict__ in = s_in + ((size_t)stage * NSEQ + s0) * ROW + jj;
      float dn_pre[SH], dz_pre[SH], dr_pre[SH], dnr[SH];
      if (unit) {
        // staged over the thread's sequences (loads, then arithmetic, then stores) for instruction-level parallelism
        float r[SH], z[SH], nn[SH], hnn[SH], hp[SH], dh[SH];
#pragma unroll
        for (int s = 0; s < SH; ++s) {
          const float* row = in + (size_t)s * ROW;
          r[s] = row[0]; z[s] = row[NU]; nn[s] = row[2 * NU]; hnn[s] = row[3 * NU];
          hp[s] = step > 0 ? row[4 * NU] : 0.f;
          dh[s] = row[5 * NU] + dprev[s];
        }
#pragma unroll
        for (int s = 0; s < SH; ++s) {
          const float dn = dh[s] * (1.f - z[s]);
          const float dz = dh[s] * (hp[s] - nn[s]);
          dn_pre[s] = dn * (1.f - nn[s] * nn[s]);
          dz_pre[s] = dz * z[s] * (1.f - z[s]);
          dr_pre[s] = dn_pre[s] * hnn[s] * r[s] * (1.f - r[s]);
          dnr[s] = dn_pre[s] * r[s];
          dhd[s] = dh[s] * z[s];
        }
#pragma unroll
        for (int s = 0; s < SH; ++s) {
          unsigned char* bp = b_seq + s * 16;
          const __nv_bfloat16 h0 = __float2bfloat16_rn(dr_pre[s]), h1 = __float2bfloat16_rn(dz_pre[s]), h2 = __float2bfloat16_rn(dnr[s]);
          *reinterpret_cast<__nv_bfloat16*>(bp + o0) = h0;
          *reinterpret_cast<__nv_bfloat16*>(bp + o1) = h1;
          *reinterpret_cast<__nv_bfloat16*>(bp + o2) = h2;
          *reinterpret_cast<__nv_bfloat16*>(bp + Cfg::B_PART + o0) = __float2bfloat16_rn(dr_pre[s] - __bfloat162float(h0));
          *reinterpret_cast<__nv_bfloat16*>(bp + Cfg::B_PART + o1) = __float2bfloat16_rn(dz_pre[s] - __bfloat162float(h1));
          *reinterpret_cast<__nv_bfloat16*>(bp + Cfg::B_PART + o2) = __float2bfloat16_rn(dnr[s] - __bfloat162float(h2));
        }
      }
      tc_fence_before();
      fence_proxy_async();
      mbar_arrive(&g_full[c]);
      mbar_arrive(&in_empty[stage]);
      // global stores after the hand-off (see the forward kernel)
      if (unit) {
#pragma unroll
        for (int s = 0; s < SH; ++s) {
          if ((valid >> s) & 1u) {
            float* g = pg[s];
            g[0] = dr_pre[s]; g[NU] = dz_pre[s]; g[2 * NU] = dn_pre[s];
            *pn[s] = dnr[s];
          }
          pg[s] += dg_stride;
          pn[s] += dn_stride;
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem, 512);
}

template <int NU>
int launch_bwd_tc(const GruBwdParams& prm, int S, cudaStream_t stream) {
  using Cfg = TcBwdCfg<NU>;
  ISA_CUDA(cudaFuncSetAttribute(gru_bwd_tc_kernel<NU>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Cfg::smem_bytes));
  dim3 grid((prm.n_seq + S - 1) / S, 2);
  gru_bwd_tc_kernel<NU><<<grid, Cfg::NT, Cfg::smem_bytes, stream>>>(prm, S);
  return ISA_OK;
}

// sequences per CTA for the tensor-core kernels: fewest waves over the SMs, then least work per step
// (S = 14 -> 148 CTAs for the 1024 rows of a batch-16 64x64 map, both directions)
int pick_S_tc(int n_seq, int num_sms) {
  const int cand[5] = {16, 14, 12, 8, 4};
  int best = 4;
  long long best_cost = -1;
  for (int c = 0; c < 5; ++c) {
    const int S = cand[c];
    const long long ctas = 2LL * ((n_seq + S - 1) / S);
    const long long waves = (ctas + num_sms - 1) / num_sms;
    const long long cost = waves * (6 + S);
    if (best_cost < 0 || cost < best_cost) { best_cost = cost; best = S; }
  }
  return best;
}

bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

size_t fwd_smem(int n, int S) { return sizeof(float) * ((size_t)n * 3 * n + 2 * (size_t)n * S); }
size_t bwd_smem(int n, int S) { return sizeof(float) * ((size_t)n * 3 * n + 3 * (size_t)n * S + (size_t)n * S); }

int pick_S(int n_seq, int num_sms) {
  // fill the machine: prefer the largest S that still gives >= ~0.8 waves of CTAs (2 directions)
  if ((long long)((n_seq + 15) / 16) * 2 * 10 >= (long long)num_sms * 8) return 16;
  if ((long long)((n_seq + 7) / 8) * 2 * 10 >= (long long)num_sms * 8) return 8;
  return 4;
}

int check_gru(int n_seq, int T, int n, int inner) {
  ISA_CHECK_ARG(n_seq > 0 && T > 0, "gru_scan: n_seq and T must be positive");
  ISA_CHECK_ARG(n >= 4 && n <= 128 && n % 4 == 0, "gru_scan: n_units must be a multiple of 4 in [4,128] (got %d)", n);
  ISA_CHECK_ARG(inner > 0, "gru_scan: inner must be positive");
  ISA_CHECK_ARG((n_seq + 3) / 4 <= 65535 * 32, "gru_scan: too many sequences");
  return ISA_OK;
}

}  // namespace

extern "C" {

int isa_gru_scan_fwd(const float* gx, const float* w_hh, const float* b_hh, const float* b_ih, int n_seq, int T, int n_units,
                     int inner, long long outer_tok_stride, long long inner_tok_stride, long long t_tok_stride,
                     float* out, float* stash, cudaStream_t stream) {
  int rc = check_gru(n_seq, T, n_units, inner);
  if (rc) return rc;
  ISA_CHECK_ARG(gx && w_hh && b_hh && out, "gru_scan_fwd: null pointer");
  IsaDeviceInfo di;
  rc = isa_device_info(&di);
  if (rc) return rc;
  GruFwdParams prm;
  prm.gx = gx; prm.w_hh = w_hh; prm.b_hh = b_hh; prm.b_ih = b_ih; prm.out = out; prm.stash = stash;
  prm.n_seq = n_seq; prm.T = T; prm.n = n_units;
  prm.map.inner = inner; prm.map.outer_stride = outer_tok_stride; prm.map.inner_stride = inner_tok_stride; prm.map.t_stride = t_tok_stride;
  if (n_units == 100 && aligned16(gx)) {
    rc = launch_fwd_tc<100>(prm, pick_S_tc(n_seq, di.num_sms), stream);
    if (rc) return rc;
    ISA_CUDA(cudaGetLastError());
    return ISA_OK;
  }
  const int S = pick_S(n_seq, di.num_sms);
  const size_t smem = fwd_smem(n_units, S);
  ISA_CHECK_ARG(smem <= (size_t)di.max_smem_optin, "gru_scan_fwd: n_units=%d needs %zu B of shared memory (> %d)", n_units, smem, di.max_smem_optin);
  const int threads = ((2 * n_units + 31) / 32) * 32;
  dim3 grid((n_seq + S - 1) / S, 2);
#define LAUNCH_FWD(SV)                                                                                          \
  {                                                                                                             \
    ISA_CUDA(cudaFuncSetAttribute(gru_scan_fwd_kernel<SV>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
    gru_scan_fwd_kernel<SV><<<grid, threads, smem, stream>>>(prm);                                              \
  }
  if (S == 16) LAUNCH_FWD(16) else if (S == 8) LAUNCH_FWD(8) else LAUNCH_FWD(4)
#undef LAUNCH_FWD
  ISA_CUDA(cudaGetLastError());
  return ISA_OK;
}

int isa_gru_scan_bwd(const float* dout, const float* out, const float* stash, const float* w_hh,
                     int n_seq, int T, int n_units,
                     int inner, long long outer_tok_stride, long long inner_tok_stride, long long t_tok_stride,
                     float* dgx, float* dghn, cudaStream_t stream) {
  int rc = check_gru(n_seq, T, n_units, inner);
  if (rc) return rc;
  ISA_CHECK_ARG(dout && out && stash && w_hh && dgx && dghn, "gru_scan_bwd: null pointer");
  IsaDeviceInfo di;
  rc = isa_device_info(&di);
  if (rc) return rc;
  GruBwdParams prm;
  prm.dout = dout; prm.out = out; prm.stash = stash; prm.w_hh = w_hh; prm.dgx = dgx; prm.dghn = dghn;
  prm.n_seq = n_seq; prm.T = T; prm.n = n_units;
  prm.map.inner = inner; prm.map.outer_stride = outer_tok_stride; prm.map.inner_stride = inner_tok_stride; prm.map.t_stride = t_tok_stride;
  if (n_units == 100 && aligned16(stash) && aligned16(out) && aligned16(dout)) {
    rc = launch_bwd_tc<100>(prm, pick_S_tc(n_seq, di.num_sms), stream);
    if (rc) return rc;
    ISA_CUDA(cudaGetLastError());
    return ISA_OK;
  }
  const int S = pick_S(n_seq, di.num_sms);
  const size_t smem = bwd_smem(n_units, S);
  ISA_CHECK_ARG(smem <= (size_t)di.max_smem_optin, "gru_scan_bwd: n_units=%d needs %zu B of shared memory (> %d)", n_units, smem, di.max_smem_optin);
  const int threads = ((2 * n_units + 31) / 32) * 32;
  dim3 grid((n_seq + S - 1) / S, 2);
#define LAUNCH_BWD(SV)                                                                                          \
  {                                                                                                             \
    ISA_CUDA(cudaFuncSetAttribute(gru_scan_bwd_kernel<SV>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
    gru_scan_bwd_kernel<SV><<<grid, threads, smem, stream>>>(prm);                                              \
  }
  if (S == 16) LAUNCH_BWD(16) else if (S == 8) LAUNCH_BWD(8) else LAUNCH_BWD(4)
#undef LAUNCH_BWD
  ISA_CUDA(cudaGetLastError());
  return ISA_OK;
}

}  // extern "C"
