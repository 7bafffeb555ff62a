// Training-set augmentation gathered from a device-resident store of decoded images (isa_b200.augment): every output
// pixel of a batch sample is pulled from its source image through an inverse affine map output -> source, written
// straight into the layouts Model.train_step reads (normalised f32 input, channels_last; u8 class map; u8 label map;
// i32 instance count).
//
//   source coordinate (exact int64, in units of 2^-33):  u = a0 (2x+1) + a1 (2y+1) + 2 a2,  v = a3 (2x+1) + a4 (2y+1) + 2 a5
//   label   = src_label[v >> 33][u >> 33], 255 outside the source                       (nearest pixel)
//   rgb     = bilinear from the four taps around (u - 2^32, v - 2^32); taps outside read 0; fp32 weights from the low
//             33 bits
//   image   = (rgb / 255 - mean) / std
//
// Three launches: the gather (with a per-sample 256-bit presence mask built by integer atomicOr, so its value does not
// depend on scheduling), the rare fallback (a sample whose view kept no instance is rendered again through the plain
// resize map), and the renumbering of the surviving ids to 0..n-1 in ascending order of the old id.  HBM-bound: 12 B
// of f32 image + 2 B of maps written per output pixel, at most 4 RGB taps + 1 label read.  No float atomics: the output
// bits do not depend on the launch order.
#include "isa_common.cuh"

namespace {

constexpr int AG_THREADS = 256;
constexpr int AG_PPT = 4;                          // output pixels per thread
constexpr int AG_TILE = AG_THREADS * AG_PPT;       // output pixels per CTA
constexpr int AG_MAX_DIM = 32767;                  // output and source sides
constexpr long long AG_COEF_LIMIT = 1LL << 44;     // |a_i| < 2^44 (|map entry| < 4096): u and v cannot overflow int64
constexpr int AG_PARAMS = 7;                       // per sample: source index, a0..a5

struct AgNorm {
  float mean[3], std[3];
};

struct AgSrc {
  long long off;
  int h, w;
  bool ok;
};

__device__ __forceinline__ AgSrc ag_src(const long long* __restrict__ store, int n_images, long long store_pixels,
                                        long long idx) {
  AgSrc s;
  s.off = 0; s.h = 0; s.w = 0; s.ok = false;
  if (idx < 0 || idx >= n_images) return s;
  const long long off = store[3 * idx], h = store[3 * idx + 1], w = store[3 * idx + 2];
  if (off < 0 || h < 1 || w < 1 || h > AG_MAX_DIM || w > AG_MAX_DIM || off > store_pixels - h * w) return s;
  s.off = off; s.h = (int)h; s.w = (int)w; s.ok = true;
  return s;
}

// the plain resize map of Prediction.image_to_tensor: a0 = round(w 2^32 / W), a4 = round(h 2^32 / H), the rest 0
// (round half up; w 2^32 / W is never exactly half-way for W < 2^32, so every rounding rule gives the same integer)
__device__ __forceinline__ void ag_plain_map(const AgSrc& s, int H, int W, long long a[6]) {
  a[0] = (((long long)s.w << 33) + W) / (2LL * W);
  a[4] = (((long long)s.h << 33) + H) / (2LL * H);
  a[1] = a[2] = a[3] = a[5] = 0;
}

__device__ __forceinline__ float ag_tap(const unsigned char* __restrict__ rgb, const AgSrc& s, long long x, long long y,
                                        int c) {
  if (x < 0 || x >= s.w || y < 0 || y >= s.h) return 0.f;
  return (float)__ldg(rgb + 3 * (s.off + y * s.w + x) + c);
}

// one output pixel; returns its (un-renumbered) label
__device__ __forceinline__ unsigned ag_pixel(const unsigned char* __restrict__ rgb, const unsigned char* __restrict__ lab,
                                             const AgSrc& s, const long long a[6], int x, int y, const AgNorm& nm,
                                             float* __restrict__ img) {
  const long long X = 2LL * x + 1, Y = 2LL * y + 1;
  const long long u = a[0] * X + a[1] * Y + 2 * a[2];
  const long long v = a[3] * X + a[4] * Y + 2 * a[5];
  const long long ix = u >> 33, iy = v >> 33;      // arithmetic shift: floor, also for negative coordinates
  unsigned l = 255u;
  if (ix >= 0 && ix < s.w && iy >= 0 && iy < s.h) l = __ldg(lab + s.off + iy * s.w + ix);
  const long long ub = u - (1LL << 32), vb = v - (1LL << 32);
  const long long x0 = ub >> 33, y0 = vb >> 33;
  const float fx = (float)(ub & ((1LL << 33) - 1)) * 0x1p-33f;
  const float fy = (float)(vb & ((1LL << 33) - 1)) * 0x1p-33f;
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    const float top = (1.f - fx) * ag_tap(rgb, s, x0, y0, c) + fx * ag_tap(rgb, s, x0 + 1, y0, c);
    const float bot = (1.f - fx) * ag_tap(rgb, s, x0, y0 + 1, c) + fx * ag_tap(rgb, s, x0 + 1, y0 + 1, c);
    const float val = (1.f - fy) * top + fy * bot;
    img[c] = (val / 255.f - nm.mean[c]) / nm.std[c];
  }
  return l;
}

// grid (tiles, b).  FALLBACK = false: render every sample through its own map, OR the ids present into mask[b].
// FALLBACK = true: only samples whose mask[b] stayed empty; render them through the plain resize map into mask2[b].
template <bool FALLBACK>
__global__ void __launch_bounds__(AG_THREADS)
augment_gather_kernel(const unsigned char* __restrict__ rgb, const unsigned char* __restrict__ lab,
                      const long long* __restrict__ store, int n_images, long long store_pixels,
                      const long long* __restrict__ params, int H, int W, AgNorm nm, float* __restrict__ image,
                      unsigned char* __restrict__ sem, unsigned char* __restrict__ ins, unsigned* __restrict__ mask,
                      unsigned* __restrict__ mask2) {
  const int b = blockIdx.y;
  if (FALLBACK) {
    unsigned any = 0;
#pragma unroll
    for (int w = 0; w < 8; ++w) any |= mask[8 * b + w];
    if (any) return;                               // uniform over the CTA
  }
  __shared__ unsigned sh_mask[8];
  if (threadIdx.x < 8) sh_mask[threadIdx.x] = 0u;
  const long long* p = params + (size_t)AG_PARAMS * b;
  const AgSrc s = ag_src(store, n_images, store_pixels, p[0]);
  long long a[6];
  bool ok = s.ok;
  if (FALLBACK) {
    ag_plain_map(s, H, W, a);
  } else {
#pragma unroll
    for (int i = 0; i < 6; ++i) {
      a[i] = p[1 + i];
      ok = ok && a[i] > -AG_COEF_LIMIT && a[i] < AG_COEF_LIMIT;
    }
  }
  unsigned m[8];
#pragma unroll
  for (int w = 0; w < 8; ++w) m[w] = 0u;
  const int HW = H * W;
  const size_t sb = (size_t)b * HW;
#pragma unroll
  for (int k = 0; k < AG_PPT; ++k) {
    const int idx = blockIdx.x * AG_TILE + k * AG_THREADS + threadIdx.x;
    if (idx >= HW) break;
    const int y = idx / W, x = idx - y * W;
    float* px = image + 3 * (sb + idx);
    unsigned l = 255u;
    if (ok) {
      l = ag_pixel(rgb, lab, s, a, x, y, nm, px);
    } else {                                       // invalid source entry or map: an empty, black sample
#pragma unroll
      for (int c = 0; c < 3; ++c) px[c] = (0.f - nm.mean[c]) / nm.std[c];
    }
    sem[sb + idx] = l != 255u;
    ins[sb + idx] = (unsigned char)l;
    if (l != 255u) {
#pragma unroll
      for (int w = 0; w < 8; ++w) m[w] |= ((int)(l >> 5) == w) ? (1u << (l & 31)) : 0u;
    }
  }
  __syncthreads();
#pragma unroll
  for (int w = 0; w < 8; ++w) {
    const unsigned r = __reduce_or_sync(0xffffffffu, m[w]);
    if ((threadIdx.x & 31) == 0 && r) atomicOr(&sh_mask[w], r);
  }
  __syncthreads();
  unsigned* out = FALLBACK ? mask2 : mask;
  if (threadIdx.x < 8 && sh_mask[threadIdx.x]) atomicOr(&out[8 * b + threadIdx.x], sh_mask[threadIdx.x]);
}

// grid (tiles, b): ids present -> 0..n-1 in ascending order; block (0, b) writes n_objects[b].  A sample whose ids are
// already 0..n-1 is left as it is.
__global__ void __launch_bounds__(AG_THREADS)
augment_renumber_kernel(int H, int W, const unsigned* __restrict__ mask, const unsigned* __restrict__ mask2,
                        unsigned char* __restrict__ ins, int* __restrict__ n_objects) {
  const int b = blockIdx.y;
  __shared__ unsigned sh_m[8];
  __shared__ unsigned char sh_map[256];
  if (threadIdx.x < 8) {
    unsigned any = 0;
    for (int w = 0; w < 8; ++w) any |= mask[8 * b + w];
    sh_m[threadIdx.x] = any ? mask[8 * b + threadIdx.x] : mask2[8 * b + threadIdx.x];
  }
  __syncthreads();
  int n = 0;
  bool compact = true;                             // ids present are exactly 0..n-1
#pragma unroll
  for (int w = 0; w < 8; ++w) {
    const unsigned mw = sh_m[w];
    n += __popc(mw);
    // compact iff every word is full until the first that is not, which is a run of low bits, and nothing follows
    compact = compact && ((mw & (mw + 1u)) == 0u) && (mw == 0u || n == 32 * w + __popc(mw));
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) n_objects[b] = n;
  if (compact) return;                             // uniform over the CTA
  {
    const int t = threadIdx.x, w = t >> 5, bit = t & 31;
    int rank = __popc(sh_m[w] & ((1u << bit) - 1u));
    for (int i = 0; i < w; ++i) rank += __popc(sh_m[i]);
    sh_map[t] = ((sh_m[w] >> bit) & 1u) ? (unsigned char)rank : (unsigned char)255;
  }
  __syncthreads();
  const int HW = H * W;
  unsigned char* ib = ins + (size_t)b * HW;
#pragma unroll
  for (int k = 0; k < AG_PPT; ++k) {
    const int idx = blockIdx.x * AG_TILE + k * AG_THREADS + threadIdx.x;
    if (idx >= HW) break;
    ib[idx] = sh_map[ib[idx]];
  }
}

}  // namespace

extern "C" size_t isa_augment_workspace_bytes(int b) {
  if (b < 1) return 0;
  return (size_t)b * 2 * 8 * sizeof(unsigned);
}

extern "C" int isa_augment(const unsigned char* rgb, const unsigned char* labels, const long long* store, int n_images,
                           long long store_pixels, const long long* params, int b, int H, int W, const float* h_mean_std,
                           float* image, unsigned char* sem, unsigned char* ins, int* n_objects, void* workspace,
                           size_t workspace_bytes, void* stream) {
  ISA_CHECK_ARG(rgb && labels && store && params && h_mean_std && image && sem && ins && n_objects && workspace,
                "isa_augment: null pointer");
  ISA_CHECK_ARG(n_images >= 1 && store_pixels >= 1, "isa_augment: n_images=%d store_pixels=%lld (both >= 1)", n_images,
                store_pixels);
  ISA_CHECK_ARG(b >= 1 && b <= 65535 && H >= 1 && W >= 1 && H <= AG_MAX_DIM && W <= AG_MAX_DIM,
                "isa_augment: b=%d H=%d W=%d (1 <= b <= 65535, 1 <= H, W <= %d)", b, H, W, AG_MAX_DIM);
  ISA_CHECK_ARG(((uintptr_t)image & 3) == 0 && ((uintptr_t)params & 7) == 0 && ((uintptr_t)store & 7) == 0 &&
                    ((uintptr_t)n_objects & 3) == 0 && ((uintptr_t)workspace & 3) == 0,
                "isa_augment: misaligned image, params, store, n_objects or workspace");
  AgNorm nm;
  for (int c = 0; c < 3; ++c) {
    nm.mean[c] = h_mean_std[c];
    nm.std[c] = h_mean_std[3 + c];
    ISA_CHECK_ARG(nm.std[c] != 0.f && nm.std[c] == nm.std[c] && nm.mean[c] == nm.mean[c],
                  "isa_augment: mean / std channel %d = %g / %g (std non-zero, both finite)", c, nm.mean[c], nm.std[c]);
  }
  const size_t need = isa_augment_workspace_bytes(b);
  if (workspace_bytes < need) {
    isa_set_error("isa_augment: workspace %zu < %zu", workspace_bytes, need);
    return ISA_ERR_WORKSPACE;
  }
  cudaStream_t st = (cudaStream_t)stream;
  unsigned* mask = (unsigned*)workspace;
  unsigned* mask2 = mask + 8 * (size_t)b;
  ISA_CUDA(cudaMemsetAsync(workspace, 0, need, st));
  const dim3 grid((unsigned)(((long long)H * W + AG_TILE - 1) / AG_TILE), (unsigned)b);
  augment_gather_kernel<false><<<grid, AG_THREADS, 0, st>>>(rgb, labels, store, n_images, store_pixels, params, H, W, nm,
                                                            image, sem, ins, mask, mask2);
  ISA_CUDA(cudaGetLastError());
  augment_gather_kernel<true><<<grid, AG_THREADS, 0, st>>>(rgb, labels, store, n_images, store_pixels, params, H, W, nm,
                                                           image, sem, ins, mask, mask2);
  ISA_CUDA(cudaGetLastError());
  augment_renumber_kernel<<<grid, AG_THREADS, 0, st>>>(H, W, mask, mask2, ins, n_objects);
  ISA_CUDA(cudaGetLastError());
  return ISA_OK;
}
