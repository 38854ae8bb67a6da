// Alpha compositing of point features along the z-sorted hits of each pixel (forward + backward).
//
// First "next" row after the rasterizer itself (SURVEY.md 8f-2; BASELINE config 3 names it): replaces
//   alphaCompositeCudaForwardKernel / alphaCompositeCudaBackwardKernel
//   (pytorch3d/csrc/compositing/alpha_composite.cu:24-70, 72-139) behind pytorch3d._C.accum_alphacomposite[_backward].
//
//   result[n,c,y,x]   = sum_k  feat[c, idx[n,k,y,x]] * cum_k * alpha[n,k,y,x],   cum_k = prod_{l<k, valid} (1 - alpha_l)
//
// Redesign: the reference runs one thread per (pixel, channel), recomputes the transmittance chain per channel,
// accumulates with atomics into a pre-zeroed result, and its backward issues O(K^2) atomics per (pixel, channel)
// on grad_alphas.  Here one thread owns a pixel: the chain is walked once, every output is written exactly once
// (no zero-fill, no atomics on result / grad_alphas), grad_alphas uses a suffix sum (O(K) per pixel, with the forward's
// front-to-back transmittance parked between its two passes), and only
// grad_features -- a genuine scatter -- uses atomics.  The forward value is bit-identical to the reference kernel:
// same products ((f * cum) * alpha), same ascending-k summation order.
// `alphas` / `points_idx` are addressed through element strides, because the renderer passes permuted views of the
// rasterizer's (N,H,W,K) outputs (pytorch3d/renderer/points/renderer.py:65-73); no copy is needed.
#include "common.cuh"
#include "raster_math.cuh"

namespace b200r {

struct Strides4 {
  int64_t n, k, y, x;
};

constexpr float kCompEps = 1e-9f;  // alpha_composite.cu:20

// The compositing backward walks a pixel's slots twice: front to back for the transmittances, back to front for the
// gradients.  Between the two passes each thread parks its pixel's transmittances in a column of shared memory when
// K <= kParkMaxK (at most 32 KB per CTA of 256; the read-back is then an on-chip load, which the `memory` clobber of
// the reductions would otherwise turn into one L2 round trip per slot), else in the slot's own gradient output.
constexpr int kParkMaxK = 32;
extern __shared__ float park_smem[];

static size_t park_smem_bytes(int K) { return K <= kParkMaxK ? (size_t)K * 256 * sizeof(float) : 0; }

// One 16-byte reduction for the four channels of a point (point-major features, C = 4): sm_90+ vector atomics.
__device__ __forceinline__ void red_add_v4(float* addr, float a, float b, float c, float d) {
  asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(addr), "f"(a), "f"(b), "f"(c), "f"(d) : "memory");
}

// Feature (c, point) lives at features[c * fs_c + point * fs_p] (the renderer passes `features_packed().permute(1, 0)`,
// a (C, P) view of point-major memory: all channels of a point in one sector, no contiguous copy).  CMAX > 0: C <= CMAX,
// the slots are walked once with one accumulator per channel -- per channel the reference's operations in its order;
// CMAX == 0: any C, channel-outer like the reference.
template <int CMAX>
__global__ void __launch_bounds__(256)
    alpha_composite_forward_kernel(const float* __restrict__ features, int64_t C, int64_t fs_c, int64_t fs_p,
                                   const float* __restrict__ alphas, Strides4 sa,
                                   const int64_t* __restrict__ points_idx, Strides4 si, int N, int K, int H, int W,
                                   float* __restrict__ result) {
  const int64_t total = (int64_t)N * H * W;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t pix = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; pix < total; pix += stride) {
    const int x = (int)(pix % W), y = (int)((pix / W) % H), n = (int)(pix / ((int64_t)W * H));
    const float* ap = alphas + n * sa.n + y * sa.y + x * sa.x;
    const int64_t* ip = points_idx + n * si.n + y * si.y + x * si.x;
    if (CMAX > 0) {
      float acc[CMAX > 0 ? CMAX : 1];
#pragma unroll
      for (int c = 0; c < CMAX; ++c) acc[c] = 0.0f;
      float cum = 1.0f;
      for (int k = 0; k < K; ++k) {
        const int64_t id = ip[k * si.k];
        if (id < 0) continue;  // -1: no point overlaps the pixel in this slot (:54-57)
        const float a = ap[k * sa.k];
#pragma unroll
        for (int c = 0; c < CMAX; ++c) {
          const float f = c < C ? __ldg(features + c * fs_c + id * fs_p) : 0.0f;
          acc[c] = fadd(acc[c], fmul(fmul(f, cum), a));  // (:63-64): features * cum_alpha * alpha
        }
        cum = fmul(cum, fsub(1.0f, a));
      }
#pragma unroll
      for (int c = 0; c < CMAX; ++c)
        if (c < C) result[(((int64_t)n * C + c) * H + y) * W + x] = acc[c];
    } else {
      for (int64_t c = 0; c < C; ++c) {
        const float* fc = features + c * fs_c;
        float acc = 0.0f, cum = 1.0f;
        for (int k = 0; k < K; ++k) {
          const int64_t id = ip[k * si.k];
          if (id < 0) continue;
          const float a = ap[k * sa.k];
          acc = fadd(acc, fmul(fmul(__ldg(fc + id * fs_p), cum), a));
          cum = fmul(cum, fsub(1.0f, a));
        }
        result[(((int64_t)n * C + c) * H + y) * W + x] = acc;
      }
    }
  }
}

__global__ void __launch_bounds__(256)
    alpha_composite_backward_kernel(const float* __restrict__ grad_out, const float* __restrict__ features, int64_t C,
                                    int64_t fs_c, int64_t fs_p, const float* __restrict__ alphas, Strides4 sa,
                                    const int64_t* __restrict__ points_idx, Strides4 si, int N, int K, int H, int W,
                                    float* __restrict__ grad_features, float* __restrict__ grad_alphas) {
  const int64_t total = (int64_t)N * H * W;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  const int64_t plane = (int64_t)H * W;
  for (int64_t pix = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; pix < total; pix += stride) {
    const int x = (int)(pix % W), y = (int)((pix / W) % H), n = (int)(pix / plane);
    const float* ap = alphas + n * sa.n + y * sa.y + x * sa.x;
    const int64_t* ip = points_idx + n * si.n + y * si.y + x * si.x;
    const float* go = grad_out + (int64_t)n * C * plane + (int64_t)y * W + x;  // + c * plane
    float* ga = grad_alphas + (int64_t)n * K * plane + (int64_t)y * W + x;     // + k * plane (contiguous N,K,H,W)
    const bool pm4 = C == 4 && fs_c == 1 && fs_p == 4 &&
                     ((reinterpret_cast<uintptr_t>(features) | reinterpret_cast<uintptr_t>(grad_features)) & 15u) == 0;
    // first pass: the transmittance in front of each valid slot, cum_k = prod_{l<k, valid} (1 - alpha_l), built front
    // to back exactly as the forward builds it and parked (see kParkMaxK; grad_alphas[k] belongs to this thread);
    // then walk the slots backwards keeping the suffix sum
    //   S_k = sum_{t>k} cum_t * alpha_t * A_t,   A_t = sum_c grad_out_c * feat[c, idx_t]
    // grad_alpha_k = cum_k * A_k - S_k / (1 - alpha_k + eps)          (alpha_composite.cu:112-134, summed over c)
    // (recovering cum_k by dividing the full product by (1 - alpha_k) loses every slot once that product underflows:
    // K = 150 at alpha 0.5, or a dozen near-opaque hits)
    float* park = K <= kParkMaxK ? park_smem + threadIdx.x : ga;
    const int64_t ps = K <= kParkMaxK ? (int64_t)blockDim.x : plane;
    float cum = 1.0f;
    for (int k = 0; k < K; ++k) {
      if (ip[k * si.k] < 0) continue;
      park[k * ps] = cum;
      cum = fmul(cum, fsub(1.0f, ap[k * sa.k]));
    }
    float suffix = 0.0f;
    for (int k = K - 1; k >= 0; --k) {
      const int64_t id = ip[k * si.k];
      if (id < 0) {
        ga[k * plane] = 0.0f;
        continue;
      }
      const float a = ap[k * sa.k];
      const float one_minus = 1.0f - a;
      const float cum_k = park[k * ps];
      float A = 0.0f;
      const float w = cum_k * a;
      if (pm4) {  // point-major features, four channels: one 16-byte load and one 16-byte reduction per hit
        const float4 f = __ldg(reinterpret_cast<const float4*>(features) + id);
        const float g0 = go[0], g1 = go[plane], g2 = go[2 * plane], g3 = go[3 * plane];
        A = ((g0 * f.x + g1 * f.y) + g2 * f.z) + g3 * f.w;
        red_add_v4(grad_features + id * 4, g0 * w, g1 * w, g2 * w, g3 * w);
      } else {
        for (int64_t c = 0; c < C; ++c) {  // (grad_features has the layout of features)
          const float g = go[c * plane];
          A += g * __ldg(features + c * fs_c + id * fs_p);
          atomicAdd(grad_features + c * fs_c + id * fs_p, g * w);  // (:115-117)
        }
      }
      ga[k * plane] = cum_k * A - suffix / (one_minus + kCompEps);
      suffix += w * A;
    }
  }
}

// ------------------------------------------------------------------------------------------------
// Weighted sum and normalised weighted sum of point features (SURVEY.md 8f-2): replace
//   weightedSumCudaForwardKernel / BackwardKernel          (pytorch3d/csrc/compositing/weighted_sum.cu:22-61, 63-103)
//   weightedSumNormCudaForwardKernel / BackwardKernel      (norm_weighted_sum.cu:24-82, 84-160)
// behind pytorch3d._C.accum_weightedsum[_backward] / accum_weightedsumnorm[_backward].
//   result[n,c,y,x] = sum_k alpha_k * feat[c, idx_k]  (/ max(sum_k alpha_k, 1e-4) when NORM)
// Same redesign as above: one thread per pixel, every output written once (the reference zero-fills `result` and
// `grad_alphas` and accumulates both with atomics, one thread per (pixel, channel)); only grad_features scatters.
// Forward: the reference's operations in its order ((f * alpha) / total, summed over ascending k) -> identical bits.
// Backward of NORM: grad_alpha_k = sum_c g_c (f_ck S - sum_t alpha_t f_ct) / S^2 = A_k / S - T / S^2 with
// A_k = sum_c g_c f_ck and T = sum_t alpha_t A_t: two passes over the K slots instead of a per-channel rescan.
// ------------------------------------------------------------------------------------------------
constexpr float kNormEps = 1e-4f;  // norm_weighted_sum.cu:20

template <bool NORM>
__global__ void __launch_bounds__(256)
    weighted_sum_forward_kernel(const float* __restrict__ features, int64_t C, int64_t P,
                                const float* __restrict__ alphas, Strides4 sa, const int64_t* __restrict__ points_idx,
                                Strides4 si, int N, int K, int H, int W, float* __restrict__ result) {
  const int64_t total = (int64_t)N * H * W;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t pix = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; pix < total; pix += stride) {
    const int x = (int)(pix % W), y = (int)((pix / W) % H), n = (int)(pix / ((int64_t)W * H));
    const float* ap = alphas + n * sa.n + y * sa.y + x * sa.x;
    const int64_t* ip = points_idx + n * si.n + y * si.y + x * si.x;
    float sum_alpha = 1.0f;
    if (NORM) {
      sum_alpha = 0.0f;
      for (int k = 0; k < K; ++k)
        if ((int)ip[k * si.k] >= 0) sum_alpha = fadd(sum_alpha, ap[k * sa.k]);  // (:54-62; index read into an int)
      if (sum_alpha < kNormEps) sum_alpha = kNormEps;
    }
    for (int64_t c = 0; c < C; ++c) {
      const float* fc = features + c * P;
      float acc = 0.0f;
      for (int k = 0; k < K; ++k) {
        const int id = (int)ip[k * si.k];
        if (id < 0) continue;
        const float t = fmul(__ldg(fc + id), ap[k * sa.k]);
        acc = fadd(acc, NORM ? fdiv(t, sum_alpha) : t);  // (norm_weighted_sum.cu:78-79, weighted_sum.cu:58)
      }
      result[(((int64_t)n * C + c) * H + y) * W + x] = acc;
    }
  }
}

template <bool NORM>
__global__ void __launch_bounds__(256)
    weighted_sum_backward_kernel(const float* __restrict__ grad_out, const float* __restrict__ features, int64_t C,
                                 int64_t P, const float* __restrict__ alphas, Strides4 sa,
                                 const int64_t* __restrict__ points_idx, Strides4 si, int N, int K, int H, int W,
                                 float* __restrict__ grad_features, float* __restrict__ grad_alphas) {
  const int64_t total = (int64_t)N * H * W;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  const int64_t plane = (int64_t)H * W;
  for (int64_t pix = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; pix < total; pix += stride) {
    const int x = (int)(pix % W), y = (int)((pix / W) % H), n = (int)(pix / plane);
    const float* ap = alphas + n * sa.n + y * sa.y + x * sa.x;
    const int64_t* ip = points_idx + n * si.n + y * si.y + x * si.x;
    const float* go = grad_out + (int64_t)n * C * plane + (int64_t)y * W + x;  // + c * plane
    float* ga = grad_alphas + (int64_t)n * K * plane + (int64_t)y * W + x;     // + k * plane (contiguous N,K,H,W)
    float S = 1.0f;
    if (NORM) {
      S = 0.0f;
      for (int k = 0; k < K; ++k)
        if ((int)ip[k * si.k] >= 0) S += ap[k * sa.k];
      if (S < kNormEps) S = kNormEps;
    }
    const float inv_s = 1.0f / S;
    float T = 0.0f;
    for (int k = 0; k < K; ++k) {
      const int id = (int)ip[k * si.k];
      if (id < 0) {
        ga[k * plane] = 0.0f;
        continue;
      }
      const float a = ap[k * sa.k];
      float A = 0.0f;
      for (int64_t c = 0; c < C; ++c) {
        const float g = go[c * plane];
        A += g * __ldg(features + c * P + id);
        atomicAdd(grad_features + c * P + id, NORM ? a * g * inv_s : a * g);  // (weighted_sum.cu:99-100, norm:155-157)
      }
      ga[k * plane] = NORM ? A * inv_s : A;
      T += a * A;
    }
    if (NORM) {
      const float corr = T * inv_s * inv_s;
      for (int k = 0; k < K; ++k)
        if ((int)ip[k * si.k] >= 0) ga[k * plane] -= corr;
    }
  }
}

// ------------------------------------------------------------------------------------------------
// Fused point rendering (optional entry point; SURVEY.md 8f-2): what PointsRenderer.forward does between the
// rasterizer and the image (pytorch3d/renderer/points/renderer.py:63-73) --
//   weights = 1 - dists / (r * r);  images = alpha_composite(idx.long().permute(0,3,1,2), weights.permute(...), features)
// -- in one kernel per direction, reading the PointFragments as the rasterizer wrote them ((N,H,W,K) int32 / float32):
// no int64 copy of the indices, no weights tensor, no permuted copies, no gradient rescaling pass (config 3: those
// element-wise passes moved 1.3 GB per step, more than the rasterizer itself).  Same operations in the same order as
// the unfused chain: 1 - d * (1.0f / r2) -- torch divides a tensor by a scalar as a product with the float reciprocal
// (BinaryDivTrueKernel.cu) -- then the reference's compositing arithmetic; the backward returns
// d loss / d dists = -(grad_alpha * (1.0f / r2)) directly.
// ------------------------------------------------------------------------------------------------
// Feature (c, point) lives at features[c * fs_c + point * fs_p]: the renderer passes `features_packed().permute(1, 0)`,
// a (C, P) VIEW of point-major memory (fs_c = 1, fs_p = C) -- all channels of a point in one sector (one 16-byte load
// when C = 4) instead of C gathers into C planes.  CMAX > 0: C <= CMAX, the slots are walked once with one accumulator
// per channel (per channel the same operations in the same order as the channel-outer loop of the reference);
// CMAX == 0: any C, channel-outer.
template <int CMAX>
__global__ void __launch_bounds__(256)
    points_alpha_render_forward_kernel(const float* __restrict__ features, int64_t C, int64_t fs_c, int64_t fs_p,
                                       const int32_t* __restrict__ idx, const float* __restrict__ dists, float r2,
                                       int N, int K, int H, int W, float* __restrict__ result) {
  const int64_t total = (int64_t)N * H * W;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  const int64_t plane = (int64_t)H * W;
  const float inv = fdiv(1.0f, r2);  // torch divides a tensor by a scalar as a product with the float reciprocal
  const bool vec4 = CMAX == 4 && C == 4 && fs_c == 1 && fs_p == 4 && (reinterpret_cast<uintptr_t>(features) & 15u) == 0;
  for (int64_t pix = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; pix < total; pix += stride) {
    const int64_t n = pix / plane, yx = pix - n * plane;
    const int32_t* ip = idx + pix * K;
    const float* dp = dists + pix * K;
    if (CMAX > 0) {
      float acc[CMAX > 0 ? CMAX : 1];
#pragma unroll
      for (int c = 0; c < CMAX; ++c) acc[c] = 0.0f;
      float cum = 1.0f;
      for (int k = 0; k < K; ++k) {
        const int id = ip[k];
        if (id < 0) continue;
        const float a = fsub(1.0f, fmul(dp[k], inv));
        float f[CMAX > 0 ? CMAX : 1];
        if (vec4) {
          const float4 v = __ldg(reinterpret_cast<const float4*>(features) + id);
          f[0] = v.x; f[1 % CMAX] = v.y; f[2 % CMAX] = v.z; f[3 % CMAX] = v.w;
        } else {
#pragma unroll
          for (int c = 0; c < CMAX; ++c) f[c] = c < C ? __ldg(features + c * fs_c + id * fs_p) : 0.0f;
        }
#pragma unroll
        for (int c = 0; c < CMAX; ++c) acc[c] = fadd(acc[c], fmul(fmul(f[c], cum), a));
        cum = fmul(cum, fsub(1.0f, a));
      }
#pragma unroll
      for (int c = 0; c < CMAX; ++c)
        if (c < C) result[(n * C + c) * plane + yx] = acc[c];
    } else {
      for (int64_t c = 0; c < C; ++c) {
        const float* fc = features + c * fs_c;
        float acc = 0.0f, cum = 1.0f;
        for (int k = 0; k < K; ++k) {
          const int id = ip[k];
          if (id < 0) continue;
          const float a = fsub(1.0f, fmul(dp[k], inv));
          acc = fadd(acc, fmul(fmul(__ldg(fc + id * fs_p), cum), a));
          cum = fmul(cum, fsub(1.0f, a));
        }
        result[(n * C + c) * plane + yx] = acc;
      }
    }
  }
}

// grad_features is addressed with the same strides as features (the caller allocates it point-major when the features
// are): the C atomics of a hit then fall into one sector.
template <int CMAX>
__global__ void __launch_bounds__(256)
    points_alpha_render_backward_kernel(const float* __restrict__ grad_out, const float* __restrict__ features,
                                        int64_t C, int64_t fs_c, int64_t fs_p, const int32_t* __restrict__ idx,
                                        const float* __restrict__ dists, float r2, int N, int K, int H, int W,
                                        float* __restrict__ grad_features, float* __restrict__ grad_dists) {
  const int64_t total = (int64_t)N * H * W;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  const int64_t plane = (int64_t)H * W;
  const float inv = fdiv(1.0f, r2);
  const bool vec4 = CMAX == 4 && C == 4 && fs_c == 1 && fs_p == 4 && (reinterpret_cast<uintptr_t>(features) & 15u) == 0;
  const bool gvec4 = (reinterpret_cast<uintptr_t>(grad_features) & 15u) == 0;
  for (int64_t pix = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; pix < total; pix += stride) {
    const int64_t n = pix / plane, yx = pix - n * plane;
    const int32_t* ip = idx + pix * K;
    const float* dp = dists + pix * K;
    const float* go = grad_out + n * C * plane + yx;  // + c * plane
    float* gd = grad_dists + pix * K;
    float g[CMAX > 0 ? CMAX : 1];
    if (CMAX > 0) {
#pragma unroll
      for (int c = 0; c < CMAX; ++c) g[c] = c < C ? go[c * plane] : 0.0f;
    }
    // (the arithmetic of alpha_composite_backward_kernel above, with alpha_k = 1 - d_k * inv; cum_k parked in shared
    // memory or in grad_dists[k] between the two passes)
    float* park = K <= kParkMaxK ? park_smem + threadIdx.x : gd;
    const int ps = K <= kParkMaxK ? (int)blockDim.x : 1;
    float cum = 1.0f;
    for (int k = 0; k < K; ++k) {
      if (ip[k] < 0) continue;
      park[k * ps] = cum;
      cum = fmul(cum, fsub(1.0f, fsub(1.0f, fmul(dp[k], inv))));
    }
    float suffix = 0.0f;
    for (int k = K - 1; k >= 0; --k) {
      const int id = ip[k];
      if (id < 0) {
        gd[k] = fmul(-0.0f, inv);
        continue;
      }
      const float a = fsub(1.0f, fmul(dp[k], inv));
      const float one_minus = 1.0f - a;
      const float cum_k = park[k * ps];
      float A = 0.0f;
      const float w = cum_k * a;
      if (CMAX > 0) {
        float f[CMAX > 0 ? CMAX : 1];
        if (vec4) {
          const float4 v = __ldg(reinterpret_cast<const float4*>(features) + id);
          f[0] = v.x; f[1 % CMAX] = v.y; f[2 % CMAX] = v.z; f[3 % CMAX] = v.w;
        } else {
#pragma unroll
          for (int c = 0; c < CMAX; ++c) f[c] = c < C ? __ldg(features + c * fs_c + id * fs_p) : 0.0f;
        }
#pragma unroll
        for (int c = 0; c < CMAX; ++c) A += g[c] * f[c];
        if (vec4 && gvec4) {
          red_add_v4(grad_features + (int64_t)id * 4, g[0] * w, g[1 % CMAX] * w, g[2 % CMAX] * w, g[3 % CMAX] * w);
        } else {
#pragma unroll
          for (int c = 0; c < CMAX; ++c)
            if (c < C) atomicAdd(grad_features + c * fs_c + id * fs_p, g[c] * w);
        }
      } else {
        for (int64_t c = 0; c < C; ++c) {
          const float gc = go[c * plane];
          A += gc * __ldg(features + c * fs_c + id * fs_p);
          atomicAdd(grad_features + c * fs_c + id * fs_p, gc * w);
        }
      }
      const float ga = cum_k * A - suffix / (one_minus + kCompEps);
      gd[k] = fmul(-ga, inv);  // d(1 - d * inv) / dd = -inv
      suffix += w * A;
    }
  }
}

}  // namespace b200r

using namespace b200r;

extern "C" int b200r_points_alpha_render_forward(const float* features, int64_t C, int64_t P,
                                                 int64_t feature_stride_c, int64_t feature_stride_p,
                                                 const int32_t* idx, const float* dists, float radius2, int32_t N,
                                                 int32_t K, int32_t H, int32_t W, float* images, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  if (C < 0 || P < 0 || N < 0 || K < 0 || H < 0 || W < 0) return fail(B200R_ERR_INVALID_ARGUMENT, "negative size");
  const int64_t total = (int64_t)N * H * W;
  if (total == 0 || C == 0) return B200R_OK;
  int64_t blocks = (total + 255) / 256;
  if (blocks > 148 * 32) blocks = 148 * 32;
#define B200R_PAR_FWD(CM)                                                                                       \
  points_alpha_render_forward_kernel<CM><<<(unsigned)blocks, 256, 0, stream>>>(                                 \
      features, C, feature_stride_c, feature_stride_p, idx, dists, radius2, N, K, H, W, images)
  if (C <= 4)
    B200R_PAR_FWD(4);
  else if (C <= 8)
    B200R_PAR_FWD(8);
  else
    B200R_PAR_FWD(0);
#undef B200R_PAR_FWD
  B200R_LAUNCHED("points_alpha_render_forward_kernel");
  return B200R_OK;
}

extern "C" int b200r_points_alpha_render_backward(const float* grad_images, const float* features, int64_t C,
                                                  int64_t P, int64_t feature_stride_c, int64_t feature_stride_p,
                                                  const int32_t* idx, const float* dists, float radius2, int32_t N,
                                                  int32_t K, int32_t H, int32_t W, float* grad_features,
                                                  float* grad_dists, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  if (C < 0 || P < 0 || N < 0 || K < 0 || H < 0 || W < 0) return fail(B200R_ERR_INVALID_ARGUMENT, "negative size");
  if (C * P > 0) B200R_CUDA_OK(cudaMemsetAsync(grad_features, 0, sizeof(float) * (size_t)(C * P), stream));
  const int64_t total = (int64_t)N * H * W;
  if (total == 0 || K == 0) return B200R_OK;
  int64_t blocks = (total + 255) / 256;
  if (blocks > 148 * 32) blocks = 148 * 32;
#define B200R_PAR_BWD(CM)                                                                                       \
  points_alpha_render_backward_kernel<CM><<<(unsigned)blocks, 256, park_smem_bytes(K), stream>>>(                                \
      grad_images, features, C, feature_stride_c, feature_stride_p, idx, dists, radius2, N, K, H, W,            \
      grad_features, grad_dists)
  if (C <= 4)
    B200R_PAR_BWD(4);
  else if (C <= 8)
    B200R_PAR_BWD(8);
  else
    B200R_PAR_BWD(0);
#undef B200R_PAR_BWD
  B200R_LAUNCHED("points_alpha_render_backward_kernel");
  return B200R_OK;
}

static int check_comp_args(int64_t C, int64_t P, int32_t N, int32_t K, int32_t H, int32_t W) {
  if (C < 0 || P < 0 || N < 0 || K < 0 || H < 0 || W < 0) return fail(B200R_ERR_INVALID_ARGUMENT, "negative size");
  return B200R_OK;
}

extern "C" int b200r_alpha_composite_forward(const float* features, int64_t C, int64_t P, const float* alphas,
                                             const int64_t* alpha_strides, const int64_t* points_idx,
                                             const int64_t* idx_strides, int32_t N, int32_t K, int32_t H, int32_t W,
                                             float* result, void* stream_) {
  return b200r_alpha_composite_forward_strided(features, C, P, P, 1, alphas, alpha_strides, points_idx, idx_strides, N,
                                               K, H, W, result, stream_);
}

extern "C" int b200r_alpha_composite_forward_strided(const float* features, int64_t C, int64_t P,
                                                     int64_t feature_stride_c, int64_t feature_stride_p,
                                                     const float* alphas, const int64_t* alpha_strides,
                                                     const int64_t* points_idx, const int64_t* idx_strides, int32_t N,
                                                     int32_t K, int32_t H, int32_t W, float* result, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  int rc = check_comp_args(C, P, N, K, H, W);
  if (rc != B200R_OK) return rc;
  const int64_t total = (int64_t)N * H * W;
  if (total == 0 || C == 0) return B200R_OK;
  const Strides4 sa = {alpha_strides[0], alpha_strides[1], alpha_strides[2], alpha_strides[3]};
  const Strides4 si = {idx_strides[0], idx_strides[1], idx_strides[2], idx_strides[3]};
  int64_t blocks = (total + 255) / 256;
  if (blocks > 148 * 32) blocks = 148 * 32;
#define B200R_AC_FWD(CM)                                                                                        \
  alpha_composite_forward_kernel<CM><<<(unsigned)blocks, 256, 0, stream>>>(                                     \
      features, C, feature_stride_c, feature_stride_p, alphas, sa, points_idx, si, N, K, H, W, result)
  if (C <= 4)
    B200R_AC_FWD(4);
  else if (C <= 8)
    B200R_AC_FWD(8);
  else
    B200R_AC_FWD(0);
#undef B200R_AC_FWD
  B200R_LAUNCHED("alpha_composite_forward_kernel");
  return B200R_OK;
}

extern "C" int b200r_alpha_composite_backward(const float* grad_out, const float* features, int64_t C, int64_t P,
                                              const float* alphas, const int64_t* alpha_strides,
                                              const int64_t* points_idx, const int64_t* idx_strides, int32_t N,
                                              int32_t K, int32_t H, int32_t W, float* grad_features,
                                              float* grad_alphas, void* stream_) {
  return b200r_alpha_composite_backward_strided(grad_out, features, C, P, P, 1, alphas, alpha_strides, points_idx,
                                                idx_strides, N, K, H, W, grad_features, grad_alphas, stream_);
}

extern "C" int b200r_alpha_composite_backward_strided(const float* grad_out, const float* features, int64_t C,
                                                      int64_t P, int64_t feature_stride_c, int64_t feature_stride_p,
                                                      const float* alphas, const int64_t* alpha_strides,
                                                      const int64_t* points_idx, const int64_t* idx_strides, int32_t N,
                                                      int32_t K, int32_t H, int32_t W, float* grad_features,
                                                      float* grad_alphas, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  int rc = check_comp_args(C, P, N, K, H, W);
  if (rc != B200R_OK) return rc;
  if (C * P > 0) B200R_CUDA_OK(cudaMemsetAsync(grad_features, 0, sizeof(float) * (size_t)(C * P), stream));
  const int64_t total = (int64_t)N * H * W;
  if (total == 0 || K == 0) return B200R_OK;
  const Strides4 sa = {alpha_strides[0], alpha_strides[1], alpha_strides[2], alpha_strides[3]};
  const Strides4 si = {idx_strides[0], idx_strides[1], idx_strides[2], idx_strides[3]};
  int64_t blocks = (total + 255) / 256;
  if (blocks > 148 * 32) blocks = 148 * 32;
  alpha_composite_backward_kernel<<<(unsigned)blocks, 256, park_smem_bytes(K), stream>>>(grad_out, features, C, feature_stride_c,
                                                                      feature_stride_p, alphas, sa, points_idx, si, N, K,
                                                                      H, W, grad_features, grad_alphas);
  B200R_LAUNCHED("alpha_composite_backward_kernel");
  return B200R_OK;
}

template <bool NORM>
static int weighted_sum_forward_impl(const float* features, int64_t C, int64_t P, const float* alphas,
                                     const int64_t* alpha_strides, const int64_t* points_idx,
                                     const int64_t* idx_strides, int32_t N, int32_t K, int32_t H, int32_t W,
                                     float* result, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  int rc = check_comp_args(C, P, N, K, H, W);
  if (rc != B200R_OK) return rc;
  const int64_t total = (int64_t)N * H * W;
  if (total == 0 || C == 0) return B200R_OK;
  const Strides4 sa = {alpha_strides[0], alpha_strides[1], alpha_strides[2], alpha_strides[3]};
  const Strides4 si = {idx_strides[0], idx_strides[1], idx_strides[2], idx_strides[3]};
  int64_t blocks = (total + 255) / 256;
  if (blocks > 148 * 32) blocks = 148 * 32;
  weighted_sum_forward_kernel<NORM><<<(unsigned)blocks, 256, 0, stream>>>(features, C, P, alphas, sa, points_idx, si, N,
                                                                        K, H, W, result);
  B200R_LAUNCHED("weighted_sum_forward_kernel");
  return B200R_OK;
}

template <bool NORM>
static int weighted_sum_backward_impl(const float* grad_out, const float* features, int64_t C, int64_t P,
                                      const float* alphas, const int64_t* alpha_strides, const int64_t* points_idx,
                                      const int64_t* idx_strides, int32_t N, int32_t K, int32_t H, int32_t W,
                                      float* grad_features, float* grad_alphas, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  int rc = check_comp_args(C, P, N, K, H, W);
  if (rc != B200R_OK) return rc;
  if (C * P > 0) B200R_CUDA_OK(cudaMemsetAsync(grad_features, 0, sizeof(float) * (size_t)(C * P), stream));
  const int64_t total = (int64_t)N * H * W;
  if (total == 0 || K == 0) return B200R_OK;
  const Strides4 sa = {alpha_strides[0], alpha_strides[1], alpha_strides[2], alpha_strides[3]};
  const Strides4 si = {idx_strides[0], idx_strides[1], idx_strides[2], idx_strides[3]};
  int64_t blocks = (total + 255) / 256;
  if (blocks > 148 * 32) blocks = 148 * 32;
  weighted_sum_backward_kernel<NORM><<<(unsigned)blocks, 256, 0, stream>>>(
      grad_out, features, C, P, alphas, sa, points_idx, si, N, K, H, W, grad_features, grad_alphas);
  B200R_LAUNCHED("weighted_sum_backward_kernel");
  return B200R_OK;
}

extern "C" int b200r_weighted_sum_forward(const float* features, int64_t C, int64_t P, const float* alphas,
                                          const int64_t* alpha_strides, const int64_t* points_idx,
                                          const int64_t* idx_strides, int32_t N, int32_t K, int32_t H, int32_t W,
                                          float* result, void* stream) {
  return weighted_sum_forward_impl<false>(features, C, P, alphas, alpha_strides, points_idx, idx_strides, N, K, H, W,
                                          result, stream);
}
extern "C" int b200r_weighted_sum_backward(const float* grad_out, const float* features, int64_t C, int64_t P,
                                           const float* alphas, const int64_t* alpha_strides,
                                           const int64_t* points_idx, const int64_t* idx_strides, int32_t N, int32_t K,
                                           int32_t H, int32_t W, float* grad_features, float* grad_alphas,
                                           void* stream) {
  return weighted_sum_backward_impl<false>(grad_out, features, C, P, alphas, alpha_strides, points_idx, idx_strides, N,
                                           K, H, W, grad_features, grad_alphas, stream);
}
extern "C" int b200r_norm_weighted_sum_forward(const float* features, int64_t C, int64_t P, const float* alphas,
                                               const int64_t* alpha_strides, const int64_t* points_idx,
                                               const int64_t* idx_strides, int32_t N, int32_t K, int32_t H, int32_t W,
                                               float* result, void* stream) {
  return weighted_sum_forward_impl<true>(features, C, P, alphas, alpha_strides, points_idx, idx_strides, N, K, H, W,
                                         result, stream);
}
extern "C" int b200r_norm_weighted_sum_backward(const float* grad_out, const float* features, int64_t C, int64_t P,
                                                const float* alphas, const int64_t* alpha_strides,
                                                const int64_t* points_idx, const int64_t* idx_strides, int32_t N,
                                                int32_t K, int32_t H, int32_t W, float* grad_features,
                                                float* grad_alphas, void* stream) {
  return weighted_sum_backward_impl<true>(grad_out, features, C, P, alphas, alpha_strides, points_idx, idx_strides, N,
                                          K, H, W, grad_features, grad_alphas, stream);
}
