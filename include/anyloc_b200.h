/*
 * anyloc_b200.h -- C ABI of libanyloc_b200.so (sm_100a).
 *
 * The reference (AnyLoc) is pure Python and has no FFI; the boundary it exposes
 * for this hot path is the Python class API of /root/reference/utilities.py.
 * Each entry point below cites the reference interface whose arithmetic it
 * replaces; the Python mirror of that API (anyloc_b200/utilities.py) binds
 * these symbols with ctypes (see INTEGRATION.md).
 *
 * Conventions: every pointer is a DEVICE pointer unless the name ends in _host;
 * every call enqueues work on `stream` (a cudaStream_t passed as void*) and
 * returns without synchronising; return value 0 = ok, negative = error (text
 * from anyloc_last_error(), thread-local).  No global state; workspaces are
 * caller-owned (sizes from the *_workspace_bytes functions).  There is NO CPU
 * fallback: without a CUDA device the compute calls return ANYLOC_ERR_CUDA.
 */
#ifndef ANYLOC_B200_H
#define ANYLOC_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ANYLOC_OK 0
#define ANYLOC_ERR_ARG (-1)
#define ANYLOC_ERR_CUDA (-2)
#define ANYLOC_ERR_WORKSPACE (-3)
#define ANYLOC_ERR_UNSUPPORTED (-4)

/* dist_mode: VLAD(dist_mode=...) utilities.py:660 */
#define ANYLOC_DIST_COSINE 0
#define ANYLOC_DIST_EUCLIDEAN 1
/* metric: get_top_k_recall(method=...) utilities.py:439-444 */
#define ANYLOC_METRIC_IP 0
#define ANYLOC_METRIC_L2 1
/* facet: DinoV2ExtractFeatures(facet=...) utilities.py:245-252,274-281 */
#define ANYLOC_FACET_QUERY 0
#define ANYLOC_FACET_KEY 1
#define ANYLOC_FACET_VALUE 2
#define ANYLOC_FACET_TOKEN 3
/* desc_mode of anyloc_vit_extract: how the selected facet rows are written */
#define ANYLOC_DESC_PLAIN 0        /* rows as computed (DinoV2ExtractFeatures norm_descs=False)                */
#define ANYLOC_DESC_L2 1           /* rows / max(|row|,1e-12)  (norm_descs=True)                              */
#define ANYLOC_DESC_INTERLEAVED 2 /* ViTExtractor layout (dino_extractor.py:329): q/k/v channel c = dd*heads + h
                                      reads projection column h*64 + dd; token rows plain; no normalisation     */
/* ffn kinds of the DINOv2 family (upstream dinov2/hub/backbones.py); DINOv1 uses ANYLOC_FFN_MLP */
#define ANYLOC_FFN_MLP 0
#define ANYLOC_FFN_SWIGLU 1

/* GEMM epilogues (internal building blocks, exported for parity tests) */
#define ANYLOC_EPI_BIAS 0          /* out = acc + bias                                   */
#define ANYLOC_EPI_BIAS_SPLIT 1    /* v = acc + bias           -> (hi,lo) tf32 pair      */
#define ANYLOC_EPI_GELU_SPLIT 2    /* v = gelu_erf(acc + bias) -> (hi,lo)                */
#define ANYLOC_EPI_SWIGLU_SPLIT 3  /* cols (2j,2j+1)=(x1,x2); v=silu(x1)*x2 -> (hi,lo)[j] */
#define ANYLOC_EPI_LS_RESID 4      /* out = resid + gamma * (acc + bias)                 */
#define ANYLOC_EPI_QKV_SPLIT 5     /* internal (ViT): q,k thirds -> (hi,lo); v third -> per-head transposed (hi,lo) */
/* GEMM input / SPLIT-output pair formats: x is carried as (hi, lo) with hi + lo ~ x to ~22 bits */
#define ANYLOC_PAIR_TF32 0         /* two fp32 arrays: hi = rna_tf32(x), lo = x - hi (kind::tf32 tensor path)          */
#define ANYLOC_PAIR_F16 1          /* two fp16 arrays of s*x (s power of two): hi = fp16(s x), lo = fp16(s x - hi);
                                      kind::f16 tensor path (2x rate); activations use s = 8, the epilogue's alpha
                                      undoes s_A*s_B.  Values beyond the fp16 range (|s x| > 65504) overflow. */
/* GEMM engines */
#define ANYLOC_GEMM_AUTO 0
#define ANYLOC_GEMM_SIMT 1         /* fp32 FFMA (validation / odd shapes)               */
#define ANYLOC_GEMM_TC3 2          /* tcgen05, 3-term split (kind::tf32 or kind::f16 by pair format) */

const char* anyloc_last_error(void);
int anyloc_version(void);
/* >0: compute capability *10 of the current device (100 on B200); <0: no usable device */
int anyloc_device_info(int* sm_count, size_t* smem_optin_bytes);

/* ------------------------------------------------------------ instrumentation (bench.py)
 * anyloc_launch_count: kernels launched by this library since load (all threads).
 * Profiling (off by default; not thread-safe): when enabled every launch group records a cudaEvent
 * pair on its stream; anyloc_profile_read synchronises them and returns, per category
 * (0 gemm_tc, 1 gemm_simt, 2 attention, 3 layernorm, 4 vit_misc, 5 vlad, 6 topk, 7 log_bin), the summed
 * device milliseconds, the number of launch groups and the summed algorithmic work
 * (FLOPs for 0-2, bytes otherwise), then clears the records. */
#define ANYLOC_PROF_CATEGORIES 8
long long anyloc_launch_count(void);
int anyloc_profile_enable(int on);
int anyloc_profile_read(double* ms, long long* groups, double* work);

/* ------------------------------------------------------------------ VLAD
 * Replaces VLAD.generate / generate_multi (utilities.py:819-926) incl. the
 * residuals of generate_res_vec (:956-962) and fpk.KMeans.predict (:849):
 *   x^ = x / max(|x|,1e-12)                (norm_descs)
 *   label = argmax_k sim(x, c_k)            (cosine: x.c_k/(|c_k|+1e-8); euclid: 2x.c_k-|c_k|^2;
 *                                            lowest k wins exact ties)
 *   V_k = sum_{label=k} (x^ - c_k);  V_k /= max(|V_k|,1e-12) (intra_norm);  V /= max(|V|,1e-12)
 * feats [B,N,D] fp32 row-major, n_valid [B] (nullable; rows >= n_valid[b] ignored, ragged lists),
 * centers [K,D], vlad [B,K*D], labels [B,N] int32 (nullable; -1 for ignored rows).
 */
size_t anyloc_vlad_workspace_bytes(int B, int N, int D, int K);
int anyloc_vlad_generate(const float* feats, const int32_t* n_valid, const float* centers,
                         int B, int N, int D, int K, int dist_mode, int norm_descs, int intra_norm,
                         float* vlad, int32_t* labels, void* ws, size_t ws_bytes, void* stream);
/* Prepared vocabulary: VLAD.generate / generate_multi are called once per image (batch) with the SAME c_centers
 * (utilities.py:216-217 of scripts/dino_v2_vlad.py fits once, then :233-237 generates for every image), so the
 * centre normalisation c/(|c|+1e-8) of fpk cos_sim, its tf32 copy and norms can be computed once.
 * anyloc_vlad_prepare fills a caller-owned device blob (anyloc_vlad_prepared_bytes); anyloc_vlad_generate_prepared
 * is anyloc_vlad_generate minus the per-call centre-prep launch.  The blob also holds a work-list counter that each
 * call leaves at zero: calls sharing a blob must be stream-ordered, and the blob must be re-prepared whenever the
 * centres (or dist_mode) change.  Results are bitwise identical to anyloc_vlad_generate. */
size_t anyloc_vlad_prepared_bytes(int D, int K);
int anyloc_vlad_prepare(const float* centers, int D, int K, int dist_mode, void* prepared, size_t prepared_bytes,
                        void* stream);
int anyloc_vlad_generate_prepared(const float* feats, const int32_t* n_valid, const float* centers, void* prepared,
                                  size_t prepared_bytes, int B, int N, int D, int K, int dist_mode, int norm_descs,
                                  int intra_norm, float* vlad, int32_t* labels, void* ws, size_t ws_bytes, void* stream);
/* Soft assignment (vlad_mode="soft", utilities.py:862-887):
 *   a[q,k] = softmax_k(soft_temp * cos(x_q, c_k))      (F.cosine_similarity :870-875, norms clamped at 1e-8)
 *   V_k    = sum_q a[q,k] * sum_c (x^_q - c_c)          (the reference weights the residuals to ALL centres by
 *                                                        cluster k's probability, :881-884)
 *   then intra / global normalisation as above.  assign [B,N,K] (nullable) receives a; padded rows get 0. */
int anyloc_vlad_generate_soft(const float* feats, const int32_t* n_valid, const float* centers,
                              int B, int N, int D, int K, float soft_temp, int norm_descs, int intra_norm,
                              float* vlad, float* assign, void* ws, size_t ws_bytes, void* stream);
/* Residual tensor of VLAD.generate_res_vec (utilities.py:928-972): out[q,k,:] = x^_q - c_k for ALL (patch, centre)
 * pairs, [N,K,D] fp32 (x^ = F.normalize(x) when norm_descs).  The reference builds every descriptor from this tensor
 * and caches it per image (`<cache_id>_r.pt`); here it is only materialised when a caller asks for it. */
int anyloc_vlad_residuals(const float* feats, const float* centers, int N, int D, int K, int norm_descs,
                          float* out, void* stream);
/* Descriptor of ONE image from a residual tensor [N,K,D] plus either the hard labels [N] int32 (utilities.py:853-861)
 * or the soft assignment [N,K] (:879-887) -- the reference's cache path (`_r.pt` + `_l.pt` / `_s.pt`, :843-852,
 * :864-878), which needs no features.  Pass exactly one of labels / assign.  vlad [K*D]. */
size_t anyloc_vlad_from_residuals_workspace_bytes(int D, int K);
int anyloc_vlad_from_residuals(const float* resid, const int32_t* labels, const float* assign, int N, int D, int K,
                               int intra_norm, float* vlad, void* ws, size_t ws_bytes, void* stream);
/* labels only (fpk.KMeans.predict, utilities.py:849; also one Lloyd assignment step of VLAD.fit :786) */
int anyloc_vlad_assign(const float* feats, const float* centers, int R, int D, int K, int dist_mode,
                       int32_t* labels, void* ws, size_t ws_bytes, void* stream);
/* one Lloyd centroid update of fpk.KMeans.fit (utilities.py:786): new_c[k] = mean of members
 * (0 for empty clusters); err_out[0] = sum((new_c - old_c)^2).  Deterministic (per-chunk partial sums added in a
 * fixed order, no floating-point atomics).  Workspace: anyloc_kmeans_workspace_bytes(R, D, K). */
size_t anyloc_kmeans_workspace_bytes(int R, int D, int K);
int anyloc_kmeans_update(const float* x, const int32_t* labels, const float* old_centers, int R, int D,
                         int K, float* new_centers, float* err_out, void* ws, size_t ws_bytes,
                         void* stream);

/* ------------------------------------------------------------- retrieval
 * Replaces the faiss part of get_top_k_recall (utilities.py:435-450): optional row
 * normalisation (F.normalize), exact inner-product / squared-L2 scores, k best per query
 * sorted best-first, lowest database index first among equal scores.
 * db [n_db,Dv], qu [n_q,Dv] fp32; dist [n_q,k] fp32; idx [n_q,k] int64.
 */
size_t anyloc_topk_workspace_bytes(int n_db, int n_q, int Dv, int k);
int anyloc_topk(const float* db, const float* qu, int n_db, int n_q, int Dv, int k, int metric,
                int normalize, float* dist, int64_t* idx, void* ws, size_t ws_bytes, void* stream);

/* Prepared database -- what `index.add(db)` leaves behind in faiss (utilities.py:449): the rows normalised (optional)
 * and stored as the (hi, lo) operand pairs the score GEMM consumes, plus |y|^2 per row (L2 metric).  Unit rows
 * (normalize != 0, Dv % 8 == 0) are kept as fp16 pairs of 4096*y (half the bytes, 2x tensor rate), other rows as tf32
 * pairs.  The blob is caller-owned (anyloc_index_bytes for `capacity` rows); rows can be added in chunks at any
 * row_offset (e.g. as descriptor batches arrive from the all-gather); a search over the first n_db rows is
 * anyloc_topk minus the per-call database pass.  `normalize` must be the same value in all calls on one blob.
 * anyloc_index_search: workspace from anyloc_index_search_workspace_bytes (query pairs + the [n_q, n_db] scores +
 * candidate lists).  Inner-product searches over an fp16-pair index run a hi-only (coarse) tensor-core pass with a
 * rigorous per-query error bound, re-score the candidates that could belong to the top-k exactly in fp32 and fall back
 * to the full 3-term product on the device when a candidate list overflows: same results, a third of the MMAs. */
size_t anyloc_index_bytes(int64_t capacity, int Dv, int normalize);
/* a fresh blob is initialised once before the first add; anyloc_index_copy moves the first n_rows rows into a larger
 * blob (growth) */
int anyloc_index_init(void* index, size_t index_bytes, int64_t capacity, int Dv, int normalize, void* stream);
int anyloc_index_copy(void* dst, size_t dst_bytes, int64_t dst_capacity, const void* src, size_t src_bytes,
                      int64_t src_capacity, int64_t n_rows, int Dv, int normalize, void* stream);
int anyloc_index_add(void* index, size_t index_bytes, int64_t capacity, int64_t row_offset, const float* rows,
                     int n_rows, int Dv, int normalize, void* stream);
size_t anyloc_index_search_workspace_bytes(int64_t n_db, int n_q, int Dv, int normalize);
int anyloc_index_search(const void* index, size_t index_bytes, int64_t capacity, int64_t n_db, const float* qu,
                        int n_q, int Dv, int k, int metric, int normalize, float* dist, int64_t* idx, void* ws,
                        size_t ws_bytes, void* stream);

/* ------------------------------------------------------------- collective
 * The one data-path collective of the pipeline (BASELINE config 4): all-gather of the [n_loc, Dv] fp32 descriptors of
 * every rank into [world * n_loc, Dv] (rank order), enqueued on `stream`.  `nccl_comm` is an ncclComm_t owned by the
 * caller (e.g. torch.distributed's NCCL backend); the library resolves ncclAllGather from the NCCL the process has
 * already loaded and returns ANYLOC_ERR_UNSUPPORTED when there is none.  The caller orders this call against its own
 * use of the communicator (one stream at a time per communicator). */
int anyloc_allgather_desc(void* nccl_comm, const float* local, float* all, size_t n_loc, int Dv, void* stream);

/* ------------------------------------------------------------------- ViT
 * Replaces DinoV2ExtractFeatures.__call__ (utilities.py:263-285) and the hub model's forward
 * it triggers (facebookresearch/dinov2 DinoVisionTransformer, see SURVEY.md App. A), with the
 * early exit at the hooked module (blocks 0..layer-1, then norm1+qkv-third or the whole block).
 * The same forward serves DINOv1 (dino_extractor.py:ViTExtractor, facebookresearch/dino): its
 * blocks are the DINOv2 MLP blocks without LayerScale (pass ones for ls1/ls2), and its patch
 * embedding may be overlapping (stride < patch).
 */
typedef struct {
  int embed_dim;   /* 384 / 768 / 1024 / 1536 */
  int depth;       /* number of blocks whose weights are supplied */
  int num_heads;   /* head_dim must be 64 */
  int ffn_kind;    /* ANYLOC_FFN_* */
  int ffn_hidden;  /* 4*D (mlp) or 4096-style fused hidden (swiglu) */
  int patch;       /* 14 (DINOv2), 8 or 16 (DINOv1) */
  int pair_dtype;  /* ANYLOC_PAIR_*: format of the weight pairs and of all GEMM-input activations */
  int stride;      /* patch-embedding conv stride: 0 = patch with H, W multiples of the patch; otherwise a divisor
                      of the patch, grid gh = 1 + (H-patch)/stride, gw = 1 + (W-patch)/stride (trailing pixels
                      dropped, like the strided Conv2d of dino_extractor.py:141-160) */
} AnylocVitCfg;

/* Per-block device pointers.  Matrices are [out,in] row-major like nn.Linear.weight, supplied as
 * tf32 (hi,lo) pairs with hi+lo == fp32 weight (anyloc_split_tf32).  For SwiGLU, w_in rows are
 * interleaved (row 2j = w12[j], row 2j+1 = w12[hidden+j]) and b_in likewise. */
typedef struct {
  const float *ln1_w, *ln1_b;
  const void *qkv_w_hi, *qkv_w_lo; const float *qkv_b;     /* [3D,D], [3D] */
  const void *proj_w_hi, *proj_w_lo; const float *proj_b;  /* [D,D],  [D]  */
  const float *ls1;                                        /* [D] LayerScale gamma */
  const float *ln2_w, *ln2_b;
  const void *in_w_hi, *in_w_lo; const float *in_b;        /* fc1 [4D,D] or interleaved w12 [2H,D] */
  const void *out_w_hi, *out_w_lo; const float *out_b;     /* fc2 [D,4D] or w3 [D,H] */
  const float *ls2;
  /* accumulator scales 1/(s_act * s_weight) of the four GEMMs (1.0 for tf32 pairs) */
  float qkv_alpha, proj_alpha, in_alpha, out_alpha;
} AnylocVitBlock;

typedef struct {
  const void *patch_w_hi, *patch_w_lo;  /* [D, Kp] conv weight flattened (c,ky,kx), zero padded to Kp */
  const float *patch_b;                 /* [D] */
  const float *cls_token;               /* [D] */
  const AnylocVitBlock* blocks;         /* HOST array [depth] of device pointers */
  float patch_alpha;
} AnylocVitWeights;

/* padded patch-embed reduction length (3*14*14=588 -> multiple of 32; 192 / 768 for patch 8 / 16) */
int anyloc_vit_patch_k(int patch);
size_t anyloc_vit_workspace_bytes(const AnylocVitCfg* cfg, int B, int H, int W);
/* img [B,3,H,W] fp32 (see AnylocVitCfg.stride for the admissible H, W); pos_embed [1+g_h*g_w, D] already
 * interpolated for this grid (upstream interpolate_pos_encoding); out [B, N(+1 if use_cls), D].
 * desc_mode: ANYLOC_DESC_* (0/1 are DinoV2ExtractFeatures' norm_descs). */
int anyloc_vit_extract(const AnylocVitCfg* cfg, const AnylocVitWeights* w_host, const float* img,
                       int B, int H, int W, const float* pos_embed, int layer, int facet,
                       int use_cls, int desc_mode, float* out, void* ws, size_t ws_bytes,
                       int gemm_engine, void* stream);

/* Log-binned descriptor of ViTExtractor._log_bin (dino_extractor.py:260-306), hierarchy 2 (the only one any
 * caller uses; others return ANYLOC_ERR_UNSUPPORTED).  x [B, gh*gw, C] fp32 (row-major grid, C % 4 == 0) ->
 * out [B, gh*gw, 17*C], bin-major (bin*C + c):
 *   bins 0-8   x  at (clamp(y+dy), clamp(x+dx)),     dy,dx in {-1,0,1} row-major
 *   bins 9-16  A1 at (clamp(y+3dy), clamp(x+3dx)),   centre skipped
 * A1 = 3x3 average, stride 1, padding 1, count_include_pad=False (AvgPool2d). */
int anyloc_log_bin(const float* x, int B, int gh, int gw, int C, int hierarchy, float* out, void* stream);

/* ------------------------------------------- building blocks (exported for parity tests)
 * C[M,N] = (A_hi+A_lo)[M,K] . (B_hi+B_lo)[N,K]^T with epilogue; *_lo nullable (treated as 0).
 * lda/ldb/ldo in elements.  out_lo/bias/gamma/resid per epilogue. */
int anyloc_gemm_nt(const void* a_hi, const void* a_lo, int lda, const void* b_hi, const void* b_lo,
                   int ldb, int M, int N, int K, int in_dtype, float alpha, int epilogue, const float* bias,
                   const float* gamma, const float* resid, void* out, void* out_lo, int ldo, int out_dtype,
                   int engine, void* stream);
int anyloc_split_tf32(const float* x, float* hi, float* lo, size_t n, void* stream);
int anyloc_split_f16(const float* x, void* hi, void* lo, size_t n, float scale, void* stream);
int anyloc_layernorm_split(const float* x, const float* w, const float* b, int M, int D, float eps,
                           void* y_hi, void* y_lo, int out_dtype, void* stream);
/* softmax(q k^T / 8) v per head (head_dim 64).  qkv (hi,lo) pairs [B,T,3D] ([q|k|v] thirds); qkv_lo may
 * be NULL for the SIMT engine (plain fp32 input).  -> o (hi,lo) [B,T,D].  engine: ANYLOC_GEMM_*. */
int anyloc_attention(const float* qkv_hi, const float* qkv_lo, int B, int T, int D, int heads,
                     void* o_hi, void* o_lo, int out_dtype, int engine, void* stream);
int anyloc_l2_normalize_rows(const float* x, int64_t rows, int D, int64_t ld_in, float* y, void* stream);

/* ------------------------------------------------------------------ sibling aggregators
 * The pooling the reference's other DINOv2 scripts apply to the same patch features [B,N,D] -> [B,D]:
 *   ANYLOC_POOL_AVG  torch.mean(ret, dim=1)        scripts/dino_v2_gp.py:130-131
 *   ANYLOC_POOL_MAX  torch.max(ret, dim=1)[0]      scripts/dino_v2_gp.py:132-133
 *   ANYLOC_POOL_GEM  m = mean(x^p) (|x|^p with gem_use_abs); sign(m)|m|^(1/p)   scripts/dino_v2_gem.py:170-189
 * n_valid [B] nullable (ragged batches). */
#define ANYLOC_POOL_AVG 0
#define ANYLOC_POOL_MAX 1
#define ANYLOC_POOL_GEM 2
int anyloc_pool(const float* feats, const int32_t* n_valid, int B, int N, int D, int mode, float gem_p,
                int gem_use_abs, float* out, void* stream);

/* ------------------------------------------------------------------ image pre-processing
 * Replaces `base_transform` (dvgl_benchmark/datasets_ws.py:20-23: T.ToTensor + T.Normalize) and the centre crop to a
 * multiple of the patch size (scripts/dino_v2_vlad.py:174-176) in one pass:
 *   out[b,c,y,x] = ((float)img[b,top+y,left+x,c] / 255 - mean[c]) / std[c]     (bit-identical to torchvision)
 * img [B,H,W,3] uint8 (device), mean3/std3 HOST arrays of 3 floats, out [B,3,Hc,Wc] fp32 (device). */
int anyloc_preprocess_u8(const uint8_t* img, int B, int H, int W, int top, int left, int Hc, int Wc,
                         const float* mean3, const float* std3, float* out, void* stream);
/* The same with the dataset loader's resize in between (dvgl_benchmark/datasets_ws.py:222-239
 * `T.functional.resize(base_transform(img), [480, 640])`; demo/anyloc_vlad_generate.py:165-177 bicubic down-scaling of
 * over-sized images): ToTensor + Normalize, ANTIALIASED resize to Hr x Wr (interpolation 0 = bilinear, 1 = bicubic --
 * torchvision's tensor defaults, i.e. torch interpolate(align_corners=False, antialias=True)), then the crop window
 * [top, top+Hc) x [left, left+Wc) of the resized image.  out [B,3,Hc,Wc]. */
int anyloc_preprocess_resize_u8(const uint8_t* img, int B, int H, int W, int Hr, int Wr, int interpolation, int top,
                                int left, int Hc, int Wc, const float* mean3, const float* std3, float* out,
                                void* stream);

#ifdef __cplusplus
}
#endif
#endif /* ANYLOC_B200_H */
