// C ABI of libanyloc_b200.so: error plumbing, building-block wrappers, GEMM engine dispatch and the
// ViT forward orchestration (early exit at the hooked module; reference
// /root/reference/utilities.py:245-252,263-285 + upstream DinoVisionTransformer for DINOv2, and
// /root/reference/dino_extractor.py:190-332 + upstream DINO VisionTransformer for DINOv1).
#include <stdarg.h>
#include <string.h>
#include <atomic>
#include <vector>
#include "epilogue.cuh"

namespace anyloc {

static thread_local char g_err[1024] = "";
void set_error(const char* fmt, ...) {
  va_list ap; va_start(ap, fmt); vsnprintf(g_err, sizeof(g_err), fmt, ap); va_end(ap);
}

static std::atomic<long long> g_launches{0};
void count_launch() { g_launches.fetch_add(1, std::memory_order_relaxed); }

namespace {
struct ProfRec { cudaEvent_t a, b; int cat; double work; };
bool g_prof_on = false;
std::vector<ProfRec> g_prof;
size_t g_prof_used = 0;
}  // namespace
ProfScope::ProfScope(int cat, cudaStream_t stream, double work) : slot(-1), st(stream) {
  if (!g_prof_on) return;
  if (g_prof_used == g_prof.size()) {
    ProfRec r{};
    if (cudaEventCreate(&r.a) != cudaSuccess || cudaEventCreate(&r.b) != cudaSuccess) return;
    g_prof.push_back(r);
  }
  slot = (int)g_prof_used++;
  g_prof[slot].cat = cat; g_prof[slot].work = work;
  cudaEventRecord(g_prof[slot].a, st);
}
ProfScope::~ProfScope() { if (slot >= 0) cudaEventRecord(g_prof[slot].b, st); }

int device_sm_count() {
  // per device ordinal: one process may drive several (possibly non-identical / MIG) devices
  static std::atomic<int> cached[64];
  int dev = 0, n = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 148;
  n = cached[dev].load(std::memory_order_relaxed);
  if (n > 0) return n;
  if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) return 148;
  cached[dev].store(n, std::memory_order_relaxed);
  return n;
}

// engines (defined in gemm_simt.cu / gemm_tc.cu)
int gemm_simt_launch(const void*, const void*, int, const void*, const void*, int, int, int, int,
                     const EpiParams&, bool f16, cudaStream_t);
int gemm_tc_launch(const void*, const void*, int, const void*, const void*, int, int, int, int,
                   const EpiParams&, bool f16, cudaStream_t);
bool gemm_tc_supported(const void* a_hi, const void* a_lo, int lda, const void* b_hi, const void* b_lo,
                       int ldb, int M, int N, int K, const EpiParams& ep, bool f16);
// vit_ops.cu / attention.cu
int launch_split(const float*, float*, float*, size_t, cudaStream_t);
int launch_split_f16(const float*, void*, void*, size_t, float, cudaStream_t);
int launch_im2col(const float*, int, int, int, int, int, int, void*, void*, bool, cudaStream_t);
int launch_assemble(const float*, const float*, const float*, int, int, int, float*, cudaStream_t);
int launch_layernorm(const float*, const float*, const float*, int, int, float, void*, void*, bool, cudaStream_t);
int launch_facet_out(const float*, int, int, int64_t, int, int, int, int, float*, cudaStream_t);
int launch_facet_interleave(const float*, int, int, int64_t, int, int, int, float*, cudaStream_t);
int launch_l2norm(const float*, int64_t, int, int64_t, float*, cudaStream_t);
int attention_launch(const float*, const float*, int, int, int, int, void*, void*, bool, cudaStream_t);
int attention_tc_launch(const float*, const float*, const float*, const float*, int, int, int, int, void*, void*, bool,
                        float*, cudaStream_t);
int attention_tc_standalone(const float*, const float*, int, int, int, int, void*, void*, bool, float*, cudaStream_t);
int attention_vt_pitch(int T);
int attention16_vt_pitch(int T);
bool attention16_vmn();
int attention_tc16_launch(const void*, const void*, const void*, const void*, int, int, int, int, void*, void*, bool,
                          cudaStream_t);
int attention_tc16_standalone(const float*, const float*, int, int, int, int, void*, void*, bool, cudaStream_t);

static int gemm_dispatch(const void* a_hi, const void* a_lo, int lda, const void* b_hi, const void* b_lo,
                         int ldb, int M, int N, int K, const EpiParams& ep, int engine, bool f16, cudaStream_t st) {
  if (M == 0 || N == 0) return ANYLOC_OK;
  bool tc_ok = gemm_tc_supported(a_hi, a_lo, lda, b_hi, b_lo, ldb, M, N, K, ep, f16);
  if (engine == ANYLOC_GEMM_TC3 && !tc_ok) {
    set_error("gemm: tcgen05 engine does not support this shape/alignment (M=%d N=%d K=%d lda=%d ldb=%d f16=%d)",
              M, N, K, lda, ldb, (int)f16);
    return ANYLOC_ERR_UNSUPPORTED;
  }
  const double flops = 2.0 * M * N * K;
  if (engine == ANYLOC_GEMM_TC3 || (engine == ANYLOC_GEMM_AUTO && tc_ok && M >= 32)) {
    ProfScope ps(PC_GEMM_TC, st, flops);
    return gemm_tc_launch(a_hi, a_lo, lda, b_hi, b_lo, ldb, M, N, K, ep, f16, st);
  }
  ProfScope ps(PC_GEMM_SIMT, st, flops);
  return gemm_simt_launch(a_hi, a_lo, lda, b_hi, b_lo, ldb, M, N, K, ep, f16, st);
}

}  // namespace anyloc

using namespace anyloc;

extern "C" const char* anyloc_last_error(void) { return g_err; }
extern "C" int anyloc_version(void) { return 100; }
extern "C" long long anyloc_launch_count(void) { return g_launches.load(); }
extern "C" int anyloc_profile_enable(int on) { g_prof_on = on != 0; g_prof_used = 0; return ANYLOC_OK; }
extern "C" int anyloc_profile_read(double* ms, long long* groups, double* work) {
  ANYLOC_REQUIRE(ms && groups && work, "profile_read: null pointer");
  for (int c = 0; c < PC_COUNT; ++c) { ms[c] = 0.0; groups[c] = 0; work[c] = 0.0; }
  for (size_t i = 0; i < g_prof_used; ++i) {
    float t = 0.f;
    ANYLOC_CHECK_CUDA(cudaEventSynchronize(g_prof[i].b));
    ANYLOC_CHECK_CUDA(cudaEventElapsedTime(&t, g_prof[i].a, g_prof[i].b));
    ms[g_prof[i].cat] += t; groups[g_prof[i].cat] += 1; work[g_prof[i].cat] += g_prof[i].work;
  }
  g_prof_used = 0;
  return ANYLOC_OK;
}

extern "C" int anyloc_device_info(int* sm_count, size_t* smem_optin_bytes) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess || n <= 0) {
    cudaGetLastError();
    set_error("no CUDA device visible (libanyloc_b200 has no CPU fallback)");
    return ANYLOC_ERR_CUDA;
  }
  int dev = 0; cudaDeviceProp p;
  ANYLOC_CHECK_CUDA(cudaGetDevice(&dev));
  ANYLOC_CHECK_CUDA(cudaGetDeviceProperties(&p, dev));
  if (sm_count) *sm_count = p.multiProcessorCount;
  if (smem_optin_bytes) *smem_optin_bytes = p.sharedMemPerBlockOptin;
  return p.major * 10 + p.minor;
}

extern "C" int anyloc_gemm_nt(const void* a_hi, const void* a_lo, int lda, const void* b_hi, const void* b_lo,
                              int ldb, int M, int N, int K, int in_dtype, float alpha, int epilogue,
                              const float* bias, const float* gamma, const float* resid, void* out, void* out_lo,
                              int ldo, int out_dtype, int engine, void* stream) {
  ANYLOC_REQUIRE(a_hi && b_hi && out, "gemm_nt: null pointer");
  ANYLOC_REQUIRE(M >= 0 && N >= 0 && K > 0, "gemm_nt: bad dims");
  ANYLOC_REQUIRE(in_dtype == ANYLOC_PAIR_TF32 || in_dtype == ANYLOC_PAIR_F16, "gemm_nt: bad in_dtype %d", in_dtype);
  ANYLOC_REQUIRE(out_dtype == ANYLOC_PAIR_TF32 || out_dtype == ANYLOC_PAIR_F16, "gemm_nt: bad out_dtype %d", out_dtype);
  ANYLOC_REQUIRE(epilogue >= ANYLOC_EPI_BIAS && epilogue <= ANYLOC_EPI_LS_RESID, "gemm_nt: bad epilogue %d", epilogue);
  if (epilogue == ANYLOC_EPI_BIAS_SPLIT || epilogue == ANYLOC_EPI_GELU_SPLIT || epilogue == ANYLOC_EPI_SWIGLU_SPLIT)
    ANYLOC_REQUIRE(out_lo, "gemm_nt: split epilogue needs out_lo");
  if (epilogue == ANYLOC_EPI_SWIGLU_SPLIT) ANYLOC_REQUIRE(N % 2 == 0, "gemm_nt: swiglu needs even N");
  if (epilogue == ANYLOC_EPI_LS_RESID) ANYLOC_REQUIRE(gamma && resid, "gemm_nt: LS_RESID needs gamma and resid");
  EpiParams ep{epilogue, bias, gamma, resid, (float*)out, (float*)out_lo, ldo};
  ep.alpha = alpha;
  ep.out_f16 = out_dtype == ANYLOC_PAIR_F16;
  return gemm_dispatch(a_hi, a_lo, lda, b_hi, b_lo, ldb, M, N, K, ep, engine, in_dtype == ANYLOC_PAIR_F16,
                       (cudaStream_t)stream);
}

// internal (topk.cu): plain-store GEMM with a device gate; not part of the public header
extern "C" int anyloc_gemm_nt_gated(const void* a_hi, const void* a_lo, int lda, const void* b_hi, const void* b_lo, int ldb,
                                    int M, int N, int K, int in_dtype, float alpha, float* out, int ldo, const int* gate,
                                    void* stream) {
  EpiParams ep{ANYLOC_EPI_BIAS, nullptr, nullptr, nullptr, out, nullptr, ldo};
  ep.alpha = alpha;
  ep.gate = gate;
  cudaStream_t st = (cudaStream_t)stream;
  const bool f16 = in_dtype == ANYLOC_PAIR_F16;
  if (gate) {      // conditional fallback: tcgen05 engine only (the gate lives in its kernels), nothing recorded
    if (!gemm_tc_supported(a_hi, a_lo, lda, b_hi, b_lo, ldb, M, N, K, ep, f16)) {
      set_error("gemm_nt_gated: shape outside the tcgen05 engine's contract");
      return ANYLOC_ERR_UNSUPPORTED;
    }
    return gemm_tc_launch(a_hi, a_lo, lda, b_hi, b_lo, ldb, M, N, K, ep, f16, st);
  }
  return gemm_dispatch(a_hi, a_lo, lda, b_hi, b_lo, ldb, M, N, K, ep, ANYLOC_GEMM_AUTO, f16, st);
}

extern "C" int anyloc_split_tf32(const float* x, float* hi, float* lo, size_t n, void* stream) {
  ANYLOC_REQUIRE(x && hi && lo, "split_tf32: null pointer");
  if (n == 0) return ANYLOC_OK;
  return launch_split(x, hi, lo, n, (cudaStream_t)stream);
}

extern "C" int anyloc_split_f16(const float* x, void* hi, void* lo, size_t n, float scale, void* stream) {
  ANYLOC_REQUIRE(x && hi && lo, "split_f16: null pointer");
  if (n == 0) return ANYLOC_OK;
  return launch_split_f16(x, hi, lo, n, scale, (cudaStream_t)stream);
}

extern "C" int anyloc_layernorm_split(const float* x, const float* w, const float* b, int M, int D,
                                      float eps, void* y_hi, void* y_lo, int out_dtype, void* stream) {
  ANYLOC_REQUIRE(x && w && b && y_hi && y_lo, "layernorm: null pointer");
  if (M == 0) return ANYLOC_OK;
  return launch_layernorm(x, w, b, M, D, eps, y_hi, y_lo, out_dtype == ANYLOC_PAIR_F16, (cudaStream_t)stream);
}

// qkv_f16: qkv_{hi,lo} already hold fp16 pairs of 8*x for all three thirds (the ViT's qkv epilogue wrote them); with
// vt_hi == nullptr the fp16 attention kernel then reads V row-major from that buffer (MN-major operand).
static int attention_dispatch(const float* qkv_hi, const float* qkv_lo, const float* vt_hi, const float* vt_lo,
                              int B, int T, int D, int heads, void* o_hi, void* o_lo, bool out_f16, int engine,
                              cudaStream_t st, bool qkv_f16 = false) {
  ProfScope ps(PC_ATTENTION, st, 4.0 * B * (double)T * T * D);
  const bool tc_ok = qkv_lo != nullptr && (D % 4) == 0 &&
                     (reinterpret_cast<uintptr_t>(qkv_hi) & 15) == 0 && (reinterpret_cast<uintptr_t>(qkv_lo) & 15) == 0;
  if (engine == ANYLOC_GEMM_TC3 && !tc_ok) {
    set_error("attention: the tcgen05 engine needs the (hi,lo) qkv pair, 16-byte aligned");
    return ANYLOC_ERR_UNSUPPORTED;
  }
  if (engine == ANYLOC_GEMM_SIMT || !tc_ok)
    return attention_launch(qkv_hi, qkv_lo, B, T, D, heads, o_hi, o_lo, out_f16, st);
  if (out_f16) {     // fp16-pair precision: operands are fp16 pairs too (inside the ViT the qkv epilogue wrote them)
    if (vt_hi || qkv_f16) return attention_tc16_launch(qkv_hi, qkv_lo, vt_hi, vt_lo, B, T, D, heads, o_hi, o_lo, true, st);
    return attention_tc16_standalone(qkv_hi, qkv_lo, B, T, D, heads, o_hi, o_lo, true, st);
  }
  if (vt_hi) return attention_tc_launch(qkv_hi, qkv_lo, vt_hi, vt_lo, B, T, D, heads, o_hi, o_lo, out_f16, nullptr, st);
  return attention_tc_standalone(qkv_hi, qkv_lo, B, T, D, heads, o_hi, o_lo, out_f16, nullptr, st);
}

extern "C" int anyloc_attention(const float* qkv_hi, const float* qkv_lo, int B, int T, int D, int heads,
                                void* o_hi, void* o_lo, int out_dtype, int engine, void* stream) {
  ANYLOC_REQUIRE(qkv_hi && o_hi && o_lo, "attention: null pointer");
  ANYLOC_REQUIRE(D == heads * 64, "attention: head_dim must be 64 (D=%d heads=%d)", D, heads);
  if (B == 0 || T == 0) return ANYLOC_OK;
  return attention_dispatch(qkv_hi, qkv_lo, nullptr, nullptr, B, T, D, heads, o_hi, o_lo,
                            out_dtype == ANYLOC_PAIR_F16, engine, (cudaStream_t)stream);
}

extern "C" int anyloc_l2_normalize_rows(const float* x, int64_t rows, int D, int64_t ld_in, float* y,
                                        void* stream) {
  ANYLOC_REQUIRE(x && y && D % 4 == 0 && ld_in % 4 == 0, "l2_normalize_rows: bad args");
  if (rows == 0) return ANYLOC_OK;
  return launch_l2norm(x, rows, D, ld_in, y, (cudaStream_t)stream);
}

// ------------------------------------------------------------------ ViT forward
extern "C" int anyloc_vit_patch_k(int patch) { return (int)align_up((size_t)3 * patch * patch, 32); }

namespace {
struct VitBuffers {
  float *pa_hi, *pa_lo, *ptmp, *x, *y_hi, *y_lo, *qkv, *qkv_lo, *vt_hi, *vt_lo, *h_hi, *h_lo;
  size_t vt_elems;
};
// patch grid of the (possibly overlapping) embedding conv: stride 0 means stride == patch
int vit_stride(const AnylocVitCfg* c) { return c->stride ? c->stride : c->patch; }
int vit_tokens(const AnylocVitCfg* c, int H, int W) {
  const int S = vit_stride(c);
  return (1 + (H - c->patch) / S) * (1 + (W - c->patch) / S);
}
size_t vit_carve(const AnylocVitCfg* c, int B, int H, int W, void* ws, size_t ws_bytes, VitBuffers* out) {
  const int P = c->patch, N = vit_tokens(c, H, W), T = N + 1, D = c->embed_dim, Kp = anyloc_vit_patch_k(P);
  const size_t M = (size_t)B * T;
  Workspace w(ws ? ws : (void*)256, ws ? ws_bytes : (size_t)-1 / 2);
  VitBuffers b;
  b.pa_hi = w.take<float>((size_t)B * N * Kp); b.pa_lo = w.take<float>((size_t)B * N * Kp);
  b.ptmp = w.take<float>((size_t)B * N * D);
  b.x = w.take<float>(M * D);
  b.y_hi = w.take<float>(M * D); b.y_lo = w.take<float>(M * D);
  b.qkv = w.take<float>(M * 3 * D); b.qkv_lo = w.take<float>(M * 3 * D);
  b.vt_elems = (size_t)B * D * attention_vt_pitch(T);
  b.vt_hi = w.take<float>(b.vt_elems); b.vt_lo = w.take<float>(b.vt_elems);
  b.h_hi = w.take<float>(M * c->ffn_hidden); b.h_lo = w.take<float>(M * c->ffn_hidden);
  if (out) *out = b;
  if (ws && (!b.pa_hi || !b.pa_lo || !b.ptmp || !b.x || !b.y_hi || !b.y_lo || !b.qkv || !b.qkv_lo || !b.vt_hi || !b.vt_lo || !b.h_hi || !b.h_lo)) return 0;
  return w.off;
}
}  // namespace

extern "C" size_t anyloc_vit_workspace_bytes(const AnylocVitCfg* cfg, int B, int H, int W) {
  if (!cfg || B <= 0 || cfg->patch <= 0 || cfg->stride < 0 || H < cfg->patch || W < cfg->patch) return 0;
  return vit_carve(cfg, B, H, W, nullptr, 0, nullptr) + 4096;
}

static int vit_block(const AnylocVitCfg* c, const AnylocVitBlock& wb, const VitBuffers& bf, int B, int T,
                     int engine, cudaStream_t st) {
  const int D = c->embed_dim, M = B * T, Hf = c->ffn_hidden;
  const bool f16 = c->pair_dtype == ANYLOC_PAIR_F16;
  int rc;
  const double ln_bytes = (f16 ? 8.0 : 12.0) * M * D;
  { ProfScope ps(PC_LAYERNORM, st, ln_bytes);
    if ((rc = launch_layernorm(bf.x, wb.ln1_w, wb.ln1_b, M, D, 1e-6f, bf.y_hi, bf.y_lo, f16, st))) return rc; }
  const bool tc_attn = engine != ANYLOC_GEMM_SIMT;
  EpiParams e_qkv{tc_attn ? ANYLOC_EPI_QKV_SPLIT : ANYLOC_EPI_BIAS_SPLIT, wb.qkv_b, nullptr, nullptr, bf.qkv,
                  bf.qkv_lo, 3 * D};
  e_qkv.vt_hi = bf.vt_hi; e_qkv.vt_lo = bf.vt_lo;
  const bool f16_attn = tc_attn && f16;       // fp16 operands for the fp16-pair precision
  e_qkv.qkv_T = T; e_qkv.qkv_Tp = f16_attn ? attention16_vt_pitch(T) : attention_vt_pitch(T); e_qkv.qkv_D = D;
  e_qkv.qkv_f16 = f16_attn;
  e_qkv.alpha = wb.qkv_alpha;
  // fp16-pair precision with the MN-major V operand: q, k AND v leave the GEMM row-major as fp16 pairs of 8*x -- the
  // plain split epilogue (fully staged, 16-byte stores); no transposed V^T copy exists
  const bool vmn = f16_attn && attention16_vmn();
  if (vmn) { e_qkv.mode = ANYLOC_EPI_BIAS_SPLIT; e_qkv.out_f16 = 1; }
  if ((rc = gemm_dispatch(bf.y_hi, bf.y_lo, D, wb.qkv_w_hi, wb.qkv_w_lo, D, M, 3 * D, D, e_qkv, engine, f16, st))) return rc;
  if ((rc = attention_dispatch(bf.qkv, bf.qkv_lo, (tc_attn && !vmn) ? bf.vt_hi : nullptr, (tc_attn && !vmn) ? bf.vt_lo : nullptr,
                               B, T, D, c->num_heads, bf.y_hi, bf.y_lo, f16, engine, st, vmn))) return rc;
  EpiParams e_proj{ANYLOC_EPI_LS_RESID, wb.proj_b, wb.ls1, bf.x, bf.x, nullptr, D};
  e_proj.alpha = wb.proj_alpha;
  if ((rc = gemm_dispatch(bf.y_hi, bf.y_lo, D, wb.proj_w_hi, wb.proj_w_lo, D, M, D, D, e_proj, engine, f16, st))) return rc;
  { ProfScope ps(PC_LAYERNORM, st, ln_bytes);
    if ((rc = launch_layernorm(bf.x, wb.ln2_w, wb.ln2_b, M, D, 1e-6f, bf.y_hi, bf.y_lo, f16, st))) return rc; }
  EpiParams e_in{c->ffn_kind == ANYLOC_FFN_MLP ? ANYLOC_EPI_GELU_SPLIT : ANYLOC_EPI_SWIGLU_SPLIT, wb.in_b, nullptr,
                 nullptr, bf.h_hi, bf.h_lo, Hf};
  e_in.alpha = wb.in_alpha; e_in.out_f16 = f16;
  const int n_in = c->ffn_kind == ANYLOC_FFN_MLP ? Hf : 2 * Hf;
  if ((rc = gemm_dispatch(bf.y_hi, bf.y_lo, D, wb.in_w_hi, wb.in_w_lo, D, M, n_in, D, e_in, engine, f16, st))) return rc;
  EpiParams e_out{ANYLOC_EPI_LS_RESID, wb.out_b, wb.ls2, bf.x, bf.x, nullptr, D};
  e_out.alpha = wb.out_alpha;
  return gemm_dispatch(bf.h_hi, bf.h_lo, Hf, wb.out_w_hi, wb.out_w_lo, Hf, M, D, Hf, e_out, engine, f16, st);
}

extern "C" int anyloc_vit_extract(const AnylocVitCfg* cfg, const AnylocVitWeights* w, const float* img,
                                  int B, int H, int W, const float* pos_embed, int layer, int facet,
                                  int use_cls, int desc_mode, float* out, void* ws, size_t ws_bytes,
                                  int gemm_engine, void* stream) {
  ANYLOC_REQUIRE(cfg && w && img && pos_embed && out && ws, "vit_extract: null pointer");
  if (cfg->stride == 0)
    ANYLOC_REQUIRE(cfg->patch > 0 && H % cfg->patch == 0 && W % cfg->patch == 0 && H > 0 && W > 0,
                   "vit_extract: H=%d W=%d must be positive multiples of the patch size %d", H, W, cfg->patch);
  else
    ANYLOC_REQUIRE(cfg->patch > 0 && cfg->stride > 0 && cfg->patch % cfg->stride == 0 && H >= cfg->patch &&
                   W >= cfg->patch, "vit_extract: stride %d must divide the patch size %d and H=%d W=%d be >= it",
                   cfg->stride, cfg->patch, H, W);
  ANYLOC_REQUIRE(desc_mode >= ANYLOC_DESC_PLAIN && desc_mode <= ANYLOC_DESC_INTERLEAVED, "vit_extract: bad desc_mode %d",
                 desc_mode);
  if (desc_mode == ANYLOC_DESC_INTERLEAVED)
    ANYLOC_REQUIRE(cfg->num_heads <= 16, "vit_extract: the interleaved layout supports at most 16 heads (got %d)",
                   cfg->num_heads);
  ANYLOC_REQUIRE(layer >= 0 && layer < cfg->depth, "vit_extract: layer %d out of range [0,%d)", layer, cfg->depth);
  ANYLOC_REQUIRE(facet >= ANYLOC_FACET_QUERY && facet <= ANYLOC_FACET_TOKEN, "vit_extract: bad facet %d", facet);
  ANYLOC_REQUIRE(cfg->embed_dim == cfg->num_heads * 64, "vit_extract: head_dim must be 64");
  ANYLOC_REQUIRE(B > 0, "vit_extract: empty batch");
  cudaStream_t st = (cudaStream_t)stream;
  const int P = cfg->patch, N = vit_tokens(cfg, H, W), T = N + 1, D = cfg->embed_dim, Kp = anyloc_vit_patch_k(P);
  const int M = B * T;
  VitBuffers bf;
  if (!vit_carve(cfg, B, H, W, ws, ws_bytes, &bf)) {
    set_error("vit_extract: workspace too small (%zu given, %zu needed)", ws_bytes,
              anyloc_vit_workspace_bytes(cfg, B, H, W));
    return ANYLOC_ERR_WORKSPACE;
  }
  int rc;
  if (gemm_engine != ANYLOC_GEMM_SIMT && !(cfg->pair_dtype == ANYLOC_PAIR_F16 && attention16_vmn()) &&
      (cfg->pair_dtype == ANYLOC_PAIR_F16 ? attention16_vt_pitch(T) != T : attention_vt_pitch(T) != T)) {
    // pad columns [T, Tp) of the transposed-V buffers are read by TMA but never written: keep them finite (zero)
    ANYLOC_CHECK_CUDA(cudaMemsetAsync(bf.vt_hi, 0, bf.vt_elems * sizeof(float), st));
    ANYLOC_CHECK_CUDA(cudaMemsetAsync(bf.vt_lo, 0, bf.vt_elems * sizeof(float), st));
  }
  const bool f16 = cfg->pair_dtype == ANYLOC_PAIR_F16;
  if ((rc = launch_im2col(img, B, H, W, P, vit_stride(cfg), Kp, bf.pa_hi, bf.pa_lo, f16, st))) return rc;
  EpiParams e_pe{ANYLOC_EPI_BIAS, w->patch_b, nullptr, nullptr, bf.ptmp, nullptr, D};
  e_pe.alpha = w->patch_alpha;
  if ((rc = gemm_dispatch(bf.pa_hi, bf.pa_lo, Kp, w->patch_w_hi, w->patch_w_lo, Kp, B * N, D, Kp, e_pe,
                          gemm_engine, f16, st))) return rc;
  if ((rc = launch_assemble(bf.ptmp, w->cls_token, pos_embed, B, N, D, bf.x, st))) return rc;
  for (int l = 0; l < layer; ++l)
    if ((rc = vit_block(cfg, w->blocks[l], bf, B, T, gemm_engine, st))) return rc;
  const AnylocVitBlock& wb = w->blocks[layer];
  if (facet == ANYLOC_FACET_TOKEN) {
    if ((rc = vit_block(cfg, wb, bf, B, T, gemm_engine, st))) return rc;
    return launch_facet_out(bf.x, B, T, D, 0, D, use_cls, desc_mode == ANYLOC_DESC_L2, out, st);
  }
  // q/k/v facet: only the requested third of the qkv projection of block `layer`
  if ((rc = launch_layernorm(bf.x, wb.ln1_w, wb.ln1_b, M, D, 1e-6f, bf.y_hi, bf.y_lo, f16, st))) return rc;
  const size_t woff = (size_t)facet * D * D * (f16 ? 2 : 4);      // bytes: weights are __half or float
  EpiParams e_f{ANYLOC_EPI_BIAS, wb.qkv_b + (size_t)facet * D, nullptr, nullptr, bf.qkv, nullptr, D};
  e_f.alpha = wb.qkv_alpha;
  if ((rc = gemm_dispatch(bf.y_hi, bf.y_lo, D, (const char*)wb.qkv_w_hi + woff,
                          (const char*)wb.qkv_w_lo + woff, D, M, D, D, e_f, gemm_engine, f16, st))) return rc;
  if (desc_mode == ANYLOC_DESC_INTERLEAVED) return launch_facet_interleave(bf.qkv, B, T, D, D, cfg->num_heads, use_cls, out, st);
  return launch_facet_out(bf.qkv, B, T, D, 0, D, use_cls, desc_mode == ANYLOC_DESC_L2, out, st);
}
