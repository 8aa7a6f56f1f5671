// Log-binned descriptors of DINOv1's ViTExtractor._log_bin (/root/reference/dino_extractor.py:260-306), hierarchy 2:
// for every grid cell (y, x) the 17 bins are
//   0-8   x  at (clamp(y+dy), clamp(x+dx)),   dy, dx in {-1, 0, 1}, row-major
//   9-16  A1 at (clamp(y+3dy), clamp(x+3dx)), same order, centre skipped
// with A1 the 3x3 AvgPool2d(stride 1, padding 1, count_include_pad=False) of x.  The output is 17x the input, so the
// kernel is bound by HBM writes: each block holds an 8x8 tile of grid cells x 32 channels plus its halo in shared
// memory, forms the 3x3 box sums there once (separably: column sums, then row sums), and streams the 17 bins out as
// 16-byte evict-first stores (8 lanes write one 128-byte run per bin and cell).
#include "common.cuh"

namespace anyloc {

namespace {
constexpr int kTile = 8;                   // grid rows and columns of the output tile
constexpr int kHaloX = 4;                  // x halo: A1 at +-3 needs x at +-4
constexpr int kXT = kTile + 2 * kHaloX;    // 16: x tile edge
constexpr int kAT = kTile + 6;             // 14: A1 tile edge (+-3)
constexpr int kCS = 32;                    // channels per block
constexpr int kC4 = kCS / 4;               // float4 lanes per cell
constexpr int kThreads = 256;
constexpr size_t kSmemBytes = sizeof(float4) * kC4 * (kXT * kXT + kAT * kXT + kAT * kAT);
}  // namespace

__global__ void __launch_bounds__(kThreads)
log_bin_kernel(const float* __restrict__ x, int gh, int gw, int C, int tiles_x, float* __restrict__ out) {
  extern __shared__ float4 lb_smem[];
  float4* xs = lb_smem;                          // [kXT][kXT][kC4]   x, zero outside the grid
  float4* vs = xs + kXT * kXT * kC4;             // [kAT][kXT][kC4]   column sums of 3 rows
  float4* as = vs + kAT * kXT * kC4;             // [kAT][kAT][kC4]   A1
  const int b = blockIdx.z, c0 = blockIdx.y * kCS;
  const int y0 = (blockIdx.x / tiles_x) * kTile, x0 = (blockIdx.x % tiles_x) * kTile;
  const int C4 = C >> 2, N = gh * gw;
  const float4* xb = reinterpret_cast<const float4*>(x) + (size_t)b * N * C4;
  const float4 zero = make_float4(0.f, 0.f, 0.f, 0.f);

  // x tile: grid rows y0-4 .. y0+11, columns x0-4 .. x0+11
  for (int i = threadIdx.x; i < kXT * kXT * kC4; i += kThreads) {
    const int q = i % kC4, cell = i / kC4, gy = y0 - kHaloX + cell / kXT, gx = x0 - kHaloX + cell % kXT;
    const int c4 = (c0 >> 2) + q;
    xs[i] = (gy >= 0 && gy < gh && gx >= 0 && gx < gw && c4 < C4) ? __ldg(xb + ((size_t)gy * gw + gx) * C4 + c4) : zero;
  }
  __syncthreads();
  // column sums over rows r-1..r+1 for A1 rows y0-3 .. y0+10 (zeros stand in for rows outside the grid)
  for (int i = threadIdx.x; i < kAT * kXT * kC4; i += kThreads) {
    const int q = i % kC4, cell = i / kC4, r = cell / kXT + 1, cx = cell % kXT;
    const float4 a = xs[((r - 1) * kXT + cx) * kC4 + q], m = xs[(r * kXT + cx) * kC4 + q],
                 c = xs[((r + 1) * kXT + cx) * kC4 + q];
    vs[i] = make_float4(a.x + m.x + c.x, a.y + m.y + c.y, a.z + m.z + c.z, a.w + m.w + c.w);
  }
  __syncthreads();
  // A1 = row sums of the column sums / number of in-grid cells of the 3x3 window
  for (int i = threadIdx.x; i < kAT * kAT * kC4; i += kThreads) {
    const int q = i % kC4, cell = i / kC4, ar = cell / kAT, ac = cell % kAT;
    const int gy = y0 - 3 + ar, gx = x0 - 3 + ac;
    if (gy < 0 || gy >= gh || gx < 0 || gx >= gw) continue;      // never read: reads are clamped into the grid
    const float cnt = (float)((min(gy + 1, gh - 1) - max(gy - 1, 0) + 1) * (min(gx + 1, gw - 1) - max(gx - 1, 0) + 1));
    const float4* v = vs + (ar * kXT + ac) * kC4 + q;      // vs columns ac..ac+2 are grid columns gx-1..gx+1
    const float4 l = v[0], m = v[kC4], r = v[2 * kC4];
    as[i] = make_float4((l.x + m.x + r.x) / cnt, (l.y + m.y + r.y) / cnt, (l.z + m.z + r.z) / cnt,
                        (l.w + m.w + r.w) / cnt);
  }
  __syncthreads();
  // 17 bins of every in-grid cell of the tile
  float4* ob = reinterpret_cast<float4*>(out) + (size_t)b * N * 17 * C4;
  const int q = threadIdx.x % kC4, c4 = (c0 >> 2) + q;
  if (c4 >= C4) return;
  for (int pb = threadIdx.x / kC4; pb < kTile * kTile * 17; pb += kThreads / kC4) {
    const int bin = pb % 17, cell = pb / 17, gy = y0 + cell / kTile, gx = x0 + cell % kTile;
    if (gy >= gh || gx >= gw) continue;
    float4 v;
    if (bin < 9) {
      const int sy = min(max(gy + bin / 3 - 1, 0), gh - 1), sx = min(max(gx + bin % 3 - 1, 0), gw - 1);
      v = xs[((sy - y0 + kHaloX) * kXT + (sx - x0 + kHaloX)) * kC4 + q];
    } else {
      const int k = bin - 9 + (bin >= 13);                  // 0..8 without the centre (4)
      const int sy = min(max(gy + 3 * (k / 3 - 1), 0), gh - 1), sx = min(max(gx + 3 * (k % 3 - 1), 0), gw - 1);
      v = as[((sy - y0 + 3) * kAT + (sx - x0 + 3)) * kC4 + q];
    }
    __stcs(ob + (((size_t)gy * gw + gx) * 17 + bin) * C4 + c4, v);
  }
}

}  // namespace anyloc

using namespace anyloc;

extern "C" int anyloc_log_bin(const float* x, int B, int gh, int gw, int C, int hierarchy, float* out, void* stream) {
  ANYLOC_REQUIRE(x && out, "log_bin: null pointer");
  if (hierarchy != 2) {
    set_error("log_bin: hierarchy %d unsupported (only 2, the value every ViTExtractor caller uses)", hierarchy);
    return ANYLOC_ERR_UNSUPPORTED;
  }
  ANYLOC_REQUIRE(B >= 0 && gh > 0 && gw > 0 && C > 0 && C % 4 == 0, "log_bin: bad shape B=%d gh=%d gw=%d C=%d", B, gh,
                 gw, C);
  ANYLOC_REQUIRE((reinterpret_cast<uintptr_t>(x) & 15) == 0 && (reinterpret_cast<uintptr_t>(out) & 15) == 0,
                 "log_bin: x and out must be 16-byte aligned");
  if (B == 0) return ANYLOC_OK;
  cudaStream_t st = (cudaStream_t)stream;
  static unsigned long long attr_seen = 0;
  if (first_use_on_this_device(&attr_seen))
    ANYLOC_CHECK_CUDA(cudaFuncSetAttribute(log_bin_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmemBytes));
  const int tiles_x = cdiv(gw, kTile);
  ANYLOC_REQUIRE(B <= 65535, "log_bin: batch %d too large", B);
  dim3 grid(tiles_x * cdiv(gh, kTile), cdiv(C, kCS), B);
  ProfScope ps(PC_LOG_BIN, st, 18.0 * 4.0 * B * (double)gh * gw * C);     // bytes: read once, write 17x
  log_bin_kernel<<<grid, kThreads, kSmemBytes, st>>>(x, gh, gw, C, tiles_x, out);
  ANYLOC_CHECK_LAUNCH();
  return ANYLOC_OK;
}
