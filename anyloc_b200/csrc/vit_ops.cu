// Element-wise / row-wise pieces of the DINOv2 forward (upstream dinov2 DinoVisionTransformer,
// reached from /root/reference/utilities.py:269): im2col for the p x p / stride s patch embedding
// (14/14 for DINOv2, 8 or 16 with stride p, p/2, p/4 for DINOv1's ViTExtractor), token assembly
// (+cls, +pos-embed), LayerNorm (eps 1e-6) fused with the tf32 (hi,lo) split that feeds the
// tensor-core GEMMs, the facet slice + F.normalize epilogue of DinoV2ExtractFeatures.__call__
// (utilities.py:270-283) and the head-interleaved facet layout of ViTExtractor.extract_descriptors
// (dino_extractor.py:329).
#include "common.cuh"

namespace anyloc {

__global__ void split_tf32_kernel(const float* __restrict__ x, float* __restrict__ hi,
                                  float* __restrict__ lo, size_t n) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  size_t stride = (size_t)gridDim.x * blockDim.x;
  for (; i < n; i += stride) { float h, l; split_tf32(x[i], h, l); hi[i] = h; lo[i] = l; }
}

// x -> fp16 pair of scale*x
__global__ void split_f16_kernel(const float* __restrict__ x, __half* __restrict__ hi, __half* __restrict__ lo,
                                 size_t n, float scale) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  size_t stride = (size_t)gridDim.x * blockDim.x;
  for (; i < n; i += stride) { __half h, l; split_f16(x[i] * scale, h, l); hi[i] = h; lo[i] = l; }
}

template <bool F16> struct PairOut;
template <> struct PairOut<false> {
  typedef float T;
  static __device__ __forceinline__ void put(float* hi, float* lo, size_t i, float v) { float h, l; split_tf32(v, h, l); hi[i] = h; lo[i] = l; }
};
template <> struct PairOut<true> {
  typedef __half T;
  static __device__ __forceinline__ void put(__half* hi, __half* lo, size_t i, float v) { __half h, l; split_f16(v * kActScale, h, l); hi[i] = h; lo[i] = l; }
};

// img [B,3,H,W] -> patches (hi,lo) [B*gh*gw, Kp], column order (c, ky, kx) like conv weight.flatten(1).
// Kernel P, stride S (S == P: the non-overlapping DINOv2 embedding), grid gh = 1 + (H-P)/S, gw = 1 + (W-P)/S.
template <bool F16>
__global__ void im2col_split_kernel(const float* __restrict__ img, int B, int H, int W, int P, int S, int Kp,
                                    typename PairOut<F16>::T* __restrict__ hi, typename PairOut<F16>::T* __restrict__ lo) {
  const int gh = 1 + (H - P) / S, gw = 1 + (W - P) / S;
  const size_t row = blockIdx.x;               // patch index
  const int b = (int)(row / (gh * gw)), pi = (int)(row % (gh * gw));
  const int py = pi / gw, px = pi % gw;
  const int Kreal = 3 * P * P;
  for (int c = threadIdx.x; c < Kp; c += blockDim.x) {
    float v = 0.f;
    if (c < Kreal) {
      int ch = c / (P * P), rem = c % (P * P), ky = rem / P, kx = rem % P;
      v = __ldg(img + (((size_t)b * 3 + ch) * H + (py * S + ky)) * W + (px * S + kx));
    }
    PairOut<F16>::put(hi, lo, row * Kp + c, v);
  }
}

// x[b,0,:] = cls + pos[0];  x[b,1+n,:] = patch[b*N+n,:] + pos[1+n]     (prepare_tokens)
__global__ void assemble_tokens_kernel(const float* __restrict__ patch, const float* __restrict__ cls,
                                       const float* __restrict__ pos, int B, int N, int D,
                                       float* __restrict__ x) {
  const size_t row = blockIdx.x;     // over B*(N+1)
  const int b = (int)(row / (N + 1)), t = (int)(row % (N + 1));
  const float* src = t == 0 ? cls : patch + ((size_t)b * N + (t - 1)) * D;
  const float* pe = pos + (size_t)t * D;
  for (int d = threadIdx.x; d < D; d += blockDim.x) x[row * D + d] = src[d] + pe[d];
}

// LayerNorm over the last dim (biased variance, eps inside sqrt) -> (hi,lo). One warp per row.
template <int MAXV, bool F16>   // float4 per lane
__global__ void __launch_bounds__(256)
layernorm_split_kernel(const float* __restrict__ x, const float* __restrict__ w,
                       const float* __restrict__ b, int M, int D, float eps,
                       typename PairOut<F16>::T* __restrict__ y_hi, typename PairOut<F16>::T* __restrict__ y_lo) {
  const int lane = threadIdx.x & 31;
  const int row = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (row >= M) return;
  const int D4 = D >> 2;
  const float4* xr = reinterpret_cast<const float4*>(x + (size_t)row * D);
  float4 v[MAXV];
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < MAXV; ++i) {
    int d = lane + i * 32;
    if (d < D4) { v[i] = xr[d]; s += (v[i].x + v[i].y) + (v[i].z + v[i].w); }
  }
  const float mean = warp_sum(s) / (float)D;
  float q = 0.f;
#pragma unroll
  for (int i = 0; i < MAXV; ++i) {
    int d = lane + i * 32;
    if (d < D4) {
      float a = v[i].x - mean, bb = v[i].y - mean, c = v[i].z - mean, e = v[i].w - mean;
      q += (a * a + bb * bb) + (c * c + e * e);
    }
  }
  const float rstd = rsqrtf(warp_sum(q) / (float)D + eps);
  const float4* w4 = reinterpret_cast<const float4*>(w);
  const float4* b4 = reinterpret_cast<const float4*>(b);
#pragma unroll
  for (int i = 0; i < MAXV; ++i) {
    int d = lane + i * 32;
    if (d < D4) {
      float4 ww = __ldg(w4 + d), bb = __ldg(b4 + d);
      const float y0 = (v[i].x - mean) * rstd * ww.x + bb.x, y1 = (v[i].y - mean) * rstd * ww.y + bb.y;
      const float y2 = (v[i].z - mean) * rstd * ww.z + bb.z, y3 = (v[i].w - mean) * rstd * ww.w + bb.w;
      if constexpr (F16) {
        uint2 h, l;
        split_f16x2(y0 * kActScale, y1 * kActScale, h.x, l.x);
        split_f16x2(y2 * kActScale, y3 * kActScale, h.y, l.y);
        reinterpret_cast<uint2*>(y_hi + (size_t)row * D)[d] = h;
        reinterpret_cast<uint2*>(y_lo + (size_t)row * D)[d] = l;
      } else {
        float4 h, l;
        split_tf32(y0, h.x, l.x); split_tf32(y1, h.y, l.y); split_tf32(y2, h.z, l.z); split_tf32(y3, h.w, l.w);
        reinterpret_cast<float4*>(y_hi + (size_t)row * D)[d] = h;
        reinterpret_cast<float4*>(y_lo + (size_t)row * D)[d] = l;
      }
    }
  }
}

// y[r,:] = x[r, 0:D] / max(|x[r]|,1e-12) (or plain copy), x rows strided by ld_in. One warp per row.
__global__ void __launch_bounds__(256)
l2norm_rows_kernel(const float* __restrict__ x, int64_t rows, int D, int64_t ld_in, int do_norm,
                   float* __restrict__ y) {
  const int lane = threadIdx.x & 31;
  const int64_t row = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (row >= rows) return;
  const float4* xr = reinterpret_cast<const float4*>(x + row * ld_in);
  float4* yr = reinterpret_cast<float4*>(y + row * D);
  const int D4 = D >> 2;
  float ss = 0.f;
  for (int d = lane; d < D4; d += 32) { float4 v = xr[d]; ss += v.x * v.x + v.y * v.y + v.z * v.z + v.w * v.w; }
  const float nrm = fmaxf(sqrtf(warp_sum(ss)), 1e-12f);
  for (int d = lane; d < D4; d += 32) {
    float4 v = xr[d];
    if (do_norm) { v.x /= nrm; v.y /= nrm; v.z /= nrm; v.w /= nrm; }
    yr[d] = v;
  }
}

// gather token rows [B, T, ld] (skipping cls unless use_cls, column offset col0) -> [B, T', D] then normalise
__global__ void __launch_bounds__(256)
facet_out_kernel(const float* __restrict__ src, int B, int T, int64_t ld, int col0, int D, int use_cls,
                 int do_norm, float* __restrict__ out) {
  const int lane = threadIdx.x & 31;
  const int Tout = use_cls ? T : T - 1;
  const int64_t row = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (row >= (int64_t)B * Tout) return;
  const int b = (int)(row / Tout), t = (int)(row % Tout) + (use_cls ? 0 : 1);
  const float4* xr = reinterpret_cast<const float4*>(src + ((int64_t)b * T + t) * ld + col0);
  float4* yr = reinterpret_cast<float4*>(out + row * D);
  const int D4 = D >> 2;
  float ss = 0.f;
  for (int d = lane; d < D4; d += 32) { float4 v = xr[d]; ss += v.x * v.x + v.y * v.y + v.z * v.z + v.w * v.w; }
  const float nrm = fmaxf(sqrtf(warp_sum(ss)), 1e-12f);
  for (int d = lane; d < D4; d += 32) {
    float4 v = xr[d];
    if (do_norm) { v.x /= nrm; v.y /= nrm; v.z /= nrm; v.w /= nrm; }
    yr[d] = v;
  }
}

// ViTExtractor's q/k/v layout: qkv[facet].permute(0,2,3,1).flatten(-2) of the [B,h,t,64] hook output puts channel
// c = dd*heads + hd at projection column hd*64 + dd.  One warp per token row: the row is read coalesced (float4) into
// shared memory as [heads][65] (the pad keeps the column gather below conflict-free), then written coalesced (float4)
// in the interleaved order.  No normalisation (extract_descriptors returns raw facets).
__global__ void __launch_bounds__(256)
facet_interleave_kernel(const float* __restrict__ src, int B, int T, int64_t ld, int D, int heads, int use_cls,
                        float* __restrict__ out) {
  extern __shared__ float sm_rows[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int Tout = use_cls ? T : T - 1;
  const int64_t row = (int64_t)blockIdx.x * 8 + warp;
  if (row >= (int64_t)B * Tout) return;
  float* s = sm_rows + warp * heads * 65;
  const int b = (int)(row / Tout), t = (int)(row % Tout) + (use_cls ? 0 : 1);
  const float4* xr = reinterpret_cast<const float4*>(src + ((int64_t)b * T + t) * ld);
  const int D4 = D >> 2;
  for (int d4 = lane; d4 < D4; d4 += 32) {
    const float4 v = xr[d4];
    const int d = d4 << 2;
    float* p = s + (d >> 6) * 65 + (d & 63);      // four columns of one head (64 % 4 == 0)
    p[0] = v.x; p[1] = v.y; p[2] = v.z; p[3] = v.w;
  }
  __syncwarp();
  float4* yr = reinterpret_cast<float4*>(out + row * D);
  for (int c4 = lane; c4 < D4; c4 += 32) {
    float r[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int c = (c4 << 2) + j, dd = c / heads, hd = c - dd * heads;
      r[j] = s[hd * 65 + dd];
    }
    yr[c4] = make_float4(r[0], r[1], r[2], r[3]);
  }
}

int launch_split(const float* x, float* hi, float* lo, size_t n, cudaStream_t st) {
  int blocks = (int)std::min<size_t>((n + 255) / 256, (size_t)device_sm_count() * 16);
  if (blocks < 1) blocks = 1;
  split_tf32_kernel<<<blocks, 256, 0, st>>>(x, hi, lo, n);
  ANYLOC_CHECK_LAUNCH();
  return ANYLOC_OK;
}
int launch_split_f16(const float* x, void* hi, void* lo, size_t n, float scale, cudaStream_t st) {
  int blocks = (int)std::min<size_t>((n + 255) / 256, (size_t)device_sm_count() * 16);
  if (blocks < 1) blocks = 1;
  split_f16_kernel<<<blocks, 256, 0, st>>>(x, (__half*)hi, (__half*)lo, n, scale);
  ANYLOC_CHECK_LAUNCH();
  return ANYLOC_OK;
}
int launch_im2col(const float* img, int B, int H, int W, int P, int S, int Kp, void* hi, void* lo, bool f16,
                  cudaStream_t st) {
  const int rows = B * (1 + (H - P) / S) * (1 + (W - P) / S);
  if (f16) im2col_split_kernel<true><<<rows, 128, 0, st>>>(img, B, H, W, P, S, Kp, (__half*)hi, (__half*)lo);
  else im2col_split_kernel<false><<<rows, 128, 0, st>>>(img, B, H, W, P, S, Kp, (float*)hi, (float*)lo);
  ANYLOC_CHECK_LAUNCH();
  return ANYLOC_OK;
}
int launch_assemble(const float* patch, const float* cls, const float* pos, int B, int N, int D, float* x,
                    cudaStream_t st) {
  assemble_tokens_kernel<<<B * (N + 1), 256, 0, st>>>(patch, cls, pos, B, N, D, x);
  ANYLOC_CHECK_LAUNCH();
  return ANYLOC_OK;
}
template <bool F16>
static void ln_launch(const float* x, const float* w, const float* b, int M, int D, float eps, void* y_hi, void* y_lo,
                      cudaStream_t st) {
  typedef typename PairOut<F16>::T T;
  int blocks = cdiv(M, 8);
  if (D <= 512) layernorm_split_kernel<4, F16><<<blocks, 256, 0, st>>>(x, w, b, M, D, eps, (T*)y_hi, (T*)y_lo);
  else if (D <= 1024) layernorm_split_kernel<8, F16><<<blocks, 256, 0, st>>>(x, w, b, M, D, eps, (T*)y_hi, (T*)y_lo);
  else layernorm_split_kernel<16, F16><<<blocks, 256, 0, st>>>(x, w, b, M, D, eps, (T*)y_hi, (T*)y_lo);
}
int launch_layernorm(const float* x, const float* w, const float* b, int M, int D, float eps, void* y_hi,
                     void* y_lo, bool f16, cudaStream_t st) {
  ANYLOC_REQUIRE(D % 4 == 0 && D <= 2048, "layernorm: D=%d unsupported (multiple of 4, <= 2048)", D);
  if (f16) ln_launch<true>(x, w, b, M, D, eps, y_hi, y_lo, st);
  else ln_launch<false>(x, w, b, M, D, eps, y_hi, y_lo, st);
  ANYLOC_CHECK_LAUNCH();
  return ANYLOC_OK;
}
int launch_facet_out(const float* src, int B, int T, int64_t ld, int col0, int D, int use_cls, int do_norm,
                     float* out, cudaStream_t st) {
  int64_t rows = (int64_t)B * (use_cls ? T : T - 1);
  facet_out_kernel<<<(int)((rows + 7) / 8), 256, 0, st>>>(src, B, T, ld, col0, D, use_cls, do_norm, out);
  ANYLOC_CHECK_LAUNCH();
  return ANYLOC_OK;
}
int launch_facet_interleave(const float* src, int B, int T, int64_t ld, int D, int heads, int use_cls, float* out,
                            cudaStream_t st) {
  int64_t rows = (int64_t)B * (use_cls ? T : T - 1);
  facet_interleave_kernel<<<(int)((rows + 7) / 8), 256, 8 * heads * 65 * sizeof(float), st>>>(src, B, T, ld, D, heads,
                                                                                              use_cls, out);
  ANYLOC_CHECK_LAUNCH();
  return ANYLOC_OK;
}
int launch_l2norm(const float* x, int64_t rows, int D, int64_t ld_in, float* y, cudaStream_t st) {
  l2norm_rows_kernel<<<(int)((rows + 7) / 8), 256, 0, st>>>(x, rows, D, ld_in, 1, y);
  ANYLOC_CHECK_LAUNCH();
  return ANYLOC_OK;
}

}  // namespace anyloc
