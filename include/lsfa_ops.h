/*
 * lsfa_ops.h - C ABI of the B200-native LSFA non-key-frame propagation path.
 *
 * Drop-in boundary for ONE path of hustvl/LSFA (dff_rfcn): compressed-stream motion
 * vectors -> stride-16 flow -> warp grid -> bilinear sample of the key-frame feature
 * -> x scale map -> (+ residual 1x1 conv) -> aggregation with the current-frame feature.
 * File:line citations are relative to the reference tree; SYM =
 * dff_rfcn/symbols/resnet_v1_101_flownet_rfcn.py.
 *
 * Conventions (mirroring how MXNet hands tensors to an operator, SURVEY.md section 8b):
 *   - every pointer is a DEVICE pointer owned by the caller; the library never
 *     allocates, frees or synchronises; work is enqueued on `stream` (a cudaStream_t
 *     passed as void*; NULL = legacy default stream) of the calling thread's current
 *     device;
 *   - return value 0 = LSFA_OK, negative = error; the message is available from the
 *     thread-local lsfa_last_error() (same shape as MXGetLastError());
 *   - `req` follows MXNet's OpReqType: 0 kNullOp (nothing is written), 1 kWriteTo,
 *     2 kWriteInplace (treated as kWriteTo), 3 kAddTo (out += result);
 *   - entry points are re-entrant: no global mutable state, safe from N host threads
 *     driving N devices (tester.py:301-309 runs one thread per GPU).
 */
#ifndef LSFA_OPS_H_
#define LSFA_OPS_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LSFA_ABI_VERSION 1

#if defined(__GNUC__)
#define LSFA_API __attribute__((visibility("default")))
#else
#define LSFA_API
#endif

/* error codes */
#define LSFA_OK             0
#define LSFA_E_BADARG     (-1)  /* NULL where a pointer is required, unknown enum value */
#define LSFA_E_SHAPE      (-2)  /* non-positive / inconsistent dimensions */
#define LSFA_E_ALIGN      (-3)  /* pointer or channel count violates a vector-width rule */
#define LSFA_E_CUDA       (-4)  /* launch failed (cudaPeekAtLastError) */
#define LSFA_E_UNSUPPORTED (-5) /* valid request this build cannot serve */

/* MXNet OpReqType */
#define LSFA_REQ_NULL    0
#define LSFA_REQ_WRITE   1
#define LSFA_REQ_INPLACE 2
#define LSFA_REQ_ADD     3

/* stride-16 reduction of the MV / residual image (lib/utils/image.py:220-222) */
#define LSFA_POOL_CENTRE2X2 0   /* what cv2.resize(fx=1/16, INTER_LINEAR) computes: parity mode */
#define LSFA_POOL_AVG16     1   /* literal 16x16 block mean */

/* where the sampling positions of the fused op come from */
#define LSFA_FLOW_PREPOOLED 0   /* flow (N,2,H,W) f32 in feature cells = `motion_vector` of SYM:571 */
#define LSFA_FLOW_RAW_I32   1   /* raw MV (N,h,w,2) int32 pixels, pooled in-kernel */
#define LSFA_FLOW_RAW_F32   2   /* raw MV (N,h,w,2) float32 pixels, pooled in-kernel */
#define LSFA_FLOW_GRID      3   /* normalised grid (N,2,H,W) f32 = output of GridGenerator */
#define LSFA_FLOW_COVIAR_I32 4  /* MV exactly as coviar returns it: (N,mv_src_h,mv_src_w,2) int32 at the
                                   video's own resolution; sign/flip (image.py:53-60), the im_scale resize
                                   (image.py:204) and the stride-16 reduction are all done in-kernel */

/* aggregation of src0 = warp(key)[*scale][+rnet(res)] with src1 = cur */
#define LSFA_W_NONE   0   /* out = src0                         (SYM:571-576, 678-680) */
#define LSFA_W_ADD    1   /* out = cur + src0                   (fuse_small_net 'add', SYM:236) */
#define LSFA_W_MEAN   2   /* out = 0.5*(src0 + cur)             (SYM:315,476) */
#define LSFA_W_LOGITS 3   /* softmax over {logit_warp, logit_cur} (Nq_net tail, SYM:104-108) */
#define LSFA_W_COSINE 4   /* logits from cosine of embeddings   (Fgfa_net, SYM:111-116,132-148) */

/* memory layout / element type of the feature tensors (key, scale_map, cur, out, emb_*) */
#define LSFA_LAYOUT_NCHW_F32  0   /* MXNet's layout: the drop-in variant */
#define LSFA_LAYOUT_NHWC_F32  1
#define LSFA_LAYOUT_NHWC_BF16 2   /* channel-vectorised fast path; fp32 accumulate */

/*
 * Argument block of the fused operator.  Zero-initialise, set struct_bytes =
 * sizeof(LsfaAggArgs), fill what the chosen modes need, leave the rest NULL/0.
 *
 *   src0[n] = BilinearSampler(key[key_index ? key_index[n] : n],
 *                             GridGenerator_warp(flow[n]))          SYM:571-572
 *             [* scale_map[n]]                                      SYM:308,470,680
 *             [+ rnet_w . res[n] + rnet_b]                          SYM:66,576
 *   out[n]  = blend(src0[n], cur[n]) by weight_mode; bypass[n] != 0 -> out[n] = cur[n]
 *             (ChooseFeat, operator_py/choose_feat.py:23-31)
 */
typedef struct LsfaAggArgs {
  int32_t struct_bytes;      /* = sizeof(LsfaAggArgs): ABI guard */
  int32_t layout;            /* LSFA_LAYOUT_* */
  int32_t N, C, H, W;        /* output frames, channels, output (= flow/grid) height, width */
  int32_t key_h, key_w;      /* spatial size of key planes; 0,0 = same as H,W */
  int32_t num_keys;          /* number of key features behind `key`; 0 = N.  key_index values are CLAMPED into
                                [0, num_keys) on the device (memory safety); the host path rejects bad slots */

  const void*    key;        /* (num_keys,C,key_h,key_w) | NHWC (num_keys,key_h,key_w,C) */
  const int32_t* key_index;  /* (N,) optional: which key feature frame n samples (tile_as.py:16-19) */

  int32_t flow_kind;         /* LSFA_FLOW_* */
  const void* flow;          /* per flow_kind */
  int32_t mv_h, mv_w;        /* raw MV image size (unpadded); H = ceil(mv_h/16), W = ceil(mv_w/16) */
  double  im_scale;          /* image.py:224: flow = pooled * im_scale / 16 */
  int32_t pool_mode;         /* LSFA_POOL_* */

  const void*  scale_map;    /* optional, same shape/layout as out */
  const float* res;          /* optional pooled residual (N,3,H,W) f32 (always NCHW) */
  const float* rnet_w;       /* (C,3) f32 = rnet_conv0 weight (C,3,1,1) */
  const float* rnet_b;       /* (C,)  f32 */

  const void*  cur;          /* same shape/layout as out; required unless weight_mode == NONE */
  int32_t weight_mode;       /* LSFA_W_* */
  const float* logits;       /* (N,2,H,W) f32: [n,0] = warp logit, [n,1] = cur logit */
  const void*  emb_warp;     /* (N,E,H,W) | NHWC (N,H,W,E): embedding of the warped feature */
  const void*  emb_cur;      /* embedding of the current feature */
  int32_t E;                 /* embedding channels (2048 in SYM:126) */
  const uint8_t* bypass;     /* (N,) optional */

  void*   out;               /* (N,C,H,W) | (N,H,W,C) */
  int32_t req;               /* LSFA_REQ_* */

  void*   workspace;         /* optional scratch of lsfa_warp_scale_aggregate_workspace_bytes() bytes:
                                required for NCHW + COSINE (per-pixel logits); otherwise it only enables
                                dynamic work claiming in the all-TMA kernels (NULL = static split; the
                                channels-last layouts need 64 bytes: one claim counter).
                                Contents need no initialisation; one workspace per in-flight call. */
  size_t  workspace_bytes;

  int32_t mv_src_h, mv_src_w; /* LSFA_FLOW_COVIAR_I32: size of the coviar image; mv_h,mv_w = cvRound(src*im_scale) */
  int32_t mv_negate;         /* LSFA_FLOW_COVIAR_I32: 1 applies motion_vector = -motion_vector (image.py:54) */
  int32_t mv_hflip;          /* LSFA_FLOW_COVIAR_I32: 1 applies the horizontal flip of image.py:56-60 */

  int32_t force_generic;     /* kernel choice (NCHW): 0 auto, 1 generic gather, 2 plane-resident LDG/STG,
                                3 all-TMA warp-specialised, 4 its experimental 2-CTA-cluster form with a multicast
                                key load (never chosen automatically); 3 and 4 fail if the kernel cannot serve the args.
                                Channels-last layouts: 0 auto (all-TMA gather-by-bulk-copy kernel where it applies),
                                1 LDG/STG tile kernel, 3 all-TMA gather-by-bulk-copy or LSFA_E_UNSUPPORTED,
                                5 window-resident all-TMA kernel on tensor maps (C * element size a multiple of 256 bytes)
                                or LSFA_E_UNSUPPORTED (never chosen automatically) */
} LsfaAggArgs;

LSFA_API int         lsfa_version(void);
LSFA_API const char* lsfa_last_error(void);   /* thread-local, never NULL */

/* a3+a5+a6 - replaces the CPU half of transform_mv_res for the MV
 * (lib/utils/image.py:207-215,220-228): zero-pad to 16, stride-16 reduction in float64,
 * times im_scale/16, HWC -> (N,2,H,W) float32 with ch0 = x, ch1 = y.
 * mv: (N,h,w,2) int32 | float32, already resized by im_scale (stage 1).  H=ceil(h/16). */
LSFA_API int lsfa_mv_pool_i32(const int32_t* mv, float* flow, int N, int h, int w,
                     double im_scale, int mode, void* stream);
LSFA_API int lsfa_mv_pool_f32(const float* mv, float* flow, int N, int h, int w,
                     double im_scale, int mode, void* stream);

/* a3+a4+a5 for the residual (image.py:207-222), including the in-place channel aliasing of
 * image.py:217-218.  res: (N,h,w,3); means: HOST pointer to 3 doubles (or NULL = zeros), pixel_scale as
 * config.network.PIXEL_MEANS / PIXEL_SCALE; out (N,3,H,W) float32. */
LSFA_API int lsfa_res_pool_i32(const int32_t* res, float* out, int N, int h, int w,
                      const double* means, double pixel_scale, int mode, void* stream);
LSFA_API int lsfa_res_pool_f32(const float* res, float* out, int N, int h, int w,
                      const double* means, double pixel_scale, int mode, void* stream);

/* a1+a2 - replaces lib/utils/image.py:52-60 (sign, optional h-flip) and :204 (cv2.resize
 * by im_scale, INTER_LINEAR, float32) for the MV.  in (N,h,w,2) int32 as coviar returns it;
 * out (N,oh,ow,2) float32 with oh = cvRound(h*im_scale).  negate=1 applies image.py:54. */
LSFA_API int lsfa_mv_prepare_i32(const int32_t* mv_coviar, float* mv_out, int N, int h, int w,
                        int oh, int ow, double im_scale, int negate, int hflip, void* stream);

/* a1+a2+a3+a4+a5 for the residual in one pass - replaces lib/utils/image.py:52,59 (the residual of
 * coviar_py2.load(...,2,True), optional h-flip), :205 (cv2.resize by im_scale, INTER_LINEAR, float32),
 * :207-215 (pad), :217-218 (aliased colour/mean loop) and :221 (stride-16 reduction).
 * res_coviar (N,h,w,3) int32 at the video's resolution; oh,ow = cvRound(h*im_scale), cvRound(w*im_scale)
 * (= h,w when im_scale == 1); means: HOST pointer to 3 doubles or NULL; out (N,3,ceil(oh/16),ceil(ow/16)) f32 =
 * the `res_diff` input of SYM:575. */
LSFA_API int lsfa_res_coviar_pool_i32(const int32_t* res_coviar, float* out, int N, int h, int w, int oh, int ow,
                             double im_scale, int hflip, const double* means, double pixel_scale, int mode,
                             void* stream);

/* Host-side helper of the reference-facing host path (lsfa_b200.host.HostAggregator; the reference copies every
 * batch host -> device in core/DataParallelExecutorGroup.py:24-39): enqueue the host -> device copy of ONLY the MV rows
 * the parity-mode reduction reads - rows 16k+7 and 16k+8 of each (h,w,2) image (lib/utils/image.py:221 as
 * LSFA_POOL_CENTRE2X2) - into the same positions of a full-size device image: 1/8 of the bytes.  mv_host: pinned host
 * memory, (N,h,w,2) 4-byte elements; mv_dev: device image of the same shape (rows never copied are never read by the
 * LSFA_FLOW_RAW_* / LSFA_POOL_CENTRE2X2 kernels).  Returns the number of bytes enqueued through *bytes_out (optional). */
LSFA_API int lsfa_mv_centre_rows_h2d(const void* mv_host, void* mv_dev, int N, int h, int w, size_t* bytes_out,
                            void* stream);

/* ---- the reference-facing HOST path: host buffers in, host buffer out ---------------------------------------
 * In the reference every forward is host -> device -> host: `_load_data` copies the batch to the GPU
 * (dff_rfcn/core/DataParallelExecutorGroup.py:24-39), the executor runs, `asnumpy()` brings the result back
 * (core/tester.py:138-145), and the key-frame feature stays ON the device between the frames of a GOP
 * (core/tester.py:246-252).  lsfa_host_aggregate_f32_nchw is that contract for the fused operator with the copies
 * explicit and overlapped: the N frames are cut into chunks, and three streams pipeline
 *     H2D(chunk i+1) | fused kernel(chunk i) | D2H(chunk i-1)
 * over `depth` staging slots.  Everything is ENQUEUED (no synchronisation): `out` is valid once stream_out has drained.
 * All host pointers must be page-locked (cudaHostAlloc / cudaHostRegister) for the copies to be asynchronous.
 * Of each (mv_h,mv_w,2) motion-vector image only the rows the stride-16 reduction reads cross PCIe
 * (lsfa_mv_centre_rows_h2d).  Device memory is the caller's: `staging` (lsfa_host_aggregate_staging_bytes, 256-byte
 * aligned, no initialisation needed, one per in-flight call sequence) and, in GOP mode, the key table.
 *
 * key_index == NULL  "private keys": key (N,C,H,W) holds one key feature per frame, uploaded with the frame.
 * key_index != NULL  "GOP mode": frame n samples key_table[key_index[n]]; the num_new_keys features in `key` are first
 *                    uploaded into slots key_slot[0..num_new_keys) of the table (the key frames that arrived with this
 *                    batch) - a key crosses PCIe once per GOP, not once per frame.  key_index / key_slot are HOST arrays. */
typedef struct LsfaHostAggArgs {
  int32_t struct_bytes;          /* = sizeof(LsfaHostAggArgs) */
  int32_t N, C, H, W;            /* frames of this call; features are NCHW float32 */
  int32_t mv_h, mv_w;            /* per-frame raw MV image (mv_h,mv_w,2) int32 at network scale (image.py:204); H = ceil(mv_h/16) */
  double  im_scale;              /* image.py:224: flow = pooled * im_scale / 16 */
  int32_t weight_mode;           /* LSFA_W_NONE | LSFA_W_ADD | LSFA_W_MEAN | LSFA_W_LOGITS */
  int32_t num_new_keys;          /* GOP mode: key features uploaded by this call (may be 0) */
  const float*   key;            /* host: (N,C,H,W) private keys | (num_new_keys,C,H,W) in GOP mode */
  const int32_t* key_slot;       /* host: (num_new_keys) */
  const int32_t* key_index;      /* host: (N) or NULL */
  const float*   scale_map;      /* host: (N,C,H,W) or NULL */
  const float*   cur;            /* host: (N,C,H,W); NULL only for LSFA_W_NONE */
  const int32_t* mv;             /* host: (N,mv_h,mv_w,2) */
  const float*   logits;         /* host: (N,2,H,W) for LSFA_W_LOGITS */
  float*         out;            /* host: (N,C,H,W) */
  float*  key_table;             /* device: (num_slots,C,H,W), GOP mode */
  int32_t num_slots;
  int32_t chunk;                 /* frames per pipeline chunk (>= 1) */
  int32_t depth;                 /* staging slots, 2..8 */
  void*   staging;               /* device scratch */
  size_t  staging_bytes;
  void*   stream_in;             /* cudaStream_t of the H2D copies   */
  void*   stream_run;            /* cudaStream_t of the fused kernel */
  void*   stream_out;            /* cudaStream_t of the D2H copies (the three may be the same stream: no overlap) */
} LsfaHostAggArgs;
LSFA_API size_t lsfa_host_aggregate_staging_bytes(const LsfaHostAggArgs* args);
LSFA_API int    lsfa_host_aggregate_f32_nchw(const LsfaHostAggArgs* args);
/* bytes one call moves over PCIe: *h2d, *d2h (either may be NULL) */
LSFA_API int    lsfa_host_aggregate_bytes(const LsfaHostAggArgs* args, size_t* h2d, size_t* d2h);

/* a7 - mx.sym.GridGenerator(data=flow, transform_type='warp') (SYM:306,320,468,571,678).
 * flow, grid: (N,2,H,W) float32. */
LSFA_API int lsfa_grid_generator_warp_f32(const float* flow, float* grid, int N, int H, int W,
                                 void* stream);

/* a8 - mx.sym.BilinearSampler(data, grid) (SYM:307,321,469,572,679).
 * data (N,C,Hi,Wi), grid (N,2,Ho,Wo) normalised to [-1,1], out (N,C,Ho,Wo); float32 NCHW. */
LSFA_API int lsfa_bilinear_sampler_f32(const float* data, const float* grid, float* out, int N, int C,
                              int Hi, int Wi, int Ho, int Wo, int req, void* stream);

/* Parity probe: the integer/indexing math of a7+a8 on its own.  From flow (N,2,H,W) (or a
 * grid when is_grid != 0) produce floor indices x0,y0 (int32) and top-left weights wx,wy
 * (float32), each (N,H,W), for a key plane of Hi x Wi. */
LSFA_API int lsfa_sampler_coords_f32(const float* flow_or_grid, int is_grid, int32_t* x0, int32_t* y0,
                            float* wx, float* wy, int N, int H, int W, int Hi, int Wi,
                            void* stream);

/* The fused operator (a5-a15 in one pass).  The two suffixed names pin the layout the
 * reference-side binding expects; lsfa_warp_scale_aggregate takes it from args->layout. */
LSFA_API int    lsfa_warp_scale_aggregate(const LsfaAggArgs* args, void* stream);
LSFA_API int    lsfa_warp_scale_aggregate_f32_nchw(const LsfaAggArgs* args, void* stream);
LSFA_API int    lsfa_warp_scale_aggregate_bf16_nhwc(const LsfaAggArgs* args, void* stream);
LSFA_API size_t lsfa_warp_scale_aggregate_workspace_bytes(const LsfaAggArgs* args);
/* kernels one call of the fused op enqueues for these args (for launch accounting) */
LSFA_API int    lsfa_warp_scale_aggregate_num_launches(const LsfaAggArgs* args);

/* a12 on its own: cosine logits of Fgfa_net (SYM:111-116,137-139).
 * emb_* (N,E,H,W) f32 (layout NCHW_F32) or (N,H,W,E) (NHWC_*); logits (N,2,H,W) f32 with
 * [n,0] = cos(emb_warp, emb_cur), [n,1] = cos(emb_cur, emb_cur). */
LSFA_API int lsfa_cosine_logits(const void* emb_warp, const void* emb_cur, float* logits, int N, int E,
                       int H, int W, int layout, void* stream);

/* Same with a caller scratch (lsfa_cosine_logits_workspace_bytes, 16-byte aligned, no initialisation): NCHW
 * embeddings then go through the all-TMA pre-pass (whole channel planes by bulk copy, per-CTA partial sums added in
 * a fixed order: deterministic); without scratch, or when the planes do not fit, this is lsfa_cosine_logits. */
LSFA_API size_t lsfa_cosine_logits_workspace_bytes(int N, int E, int H, int W, int layout);
LSFA_API int lsfa_cosine_logits_ws(const void* emb_warp, const void* emb_cur, float* logits, int N, int E, int H, int W,
                                   int layout, void* workspace, size_t workspace_bytes, void* stream);

/* Backward of the NCHW float32 cosine logits (lsfa_cosine_logits_ws): from grad_logits (N,2,H,W) = d/d(logits) to
 * grad_emb_warp, grad_emb_cur (N,E,H,W).  The logits are recomputed with the forward's kernel and summation order
 * (the all-TMA pre-pass where lsfa_cosine_logits_ws with its full workspace runs it, else the LDG kernel), then one
 * pass over both embeddings writes both gradients; no atomics, the results are the same bits run to run.
 * req_* follow OpReqType (kNullOp or a NULL pointer skips that gradient).  The gradients must not overlap the inputs
 * or each other.  workspace: lsfa_cosine_logits_backward_workspace_bytes, 16-byte aligned, no initialisation needed.
 * kernel: 0 auto, 1 the plain LDG/STG kernel, 2 the all-TMA kernel (LSFA_E_UNSUPPORTED where it cannot serve the
 * arguments: planes above 4,320 pixels, odd E or H*W, pointers not 16-byte aligned).  Both give the same bits. */
LSFA_API size_t lsfa_cosine_logits_backward_workspace_bytes(int N, int E, int H, int W);
LSFA_API int lsfa_cosine_logits_backward_f32_nchw(const float* emb_warp, const float* emb_cur, const float* grad_logits,
                                                  float* grad_emb_warp, float* grad_emb_cur, int N, int E, int H, int W,
                                                  int req_warp, int req_cur, void* workspace, size_t workspace_bytes,
                                                  int kernel, void* stream);

/* The reference graph op by op (one kernel per MXNet operator, each a full pass over
 * HBM) - the "unfused" arm of the ablation; same results as the fused op in LOGITS mode
 * with scale_map.  tmp: 5 feature-sized float32 buffers (N*C*H*W each), caller-owned. */
LSFA_API int lsfa_unfused_chain_f32_nchw(const float* key, const float* flow, const float* scale_map,
                                const float* cur, const float* logits, float* out, float* tmp,
                                int N, int C, int H, int W, void* stream);
LSFA_API int lsfa_unfused_chain_num_launches(void);

/* a12/a13 tail on its own (SYM:104-108, 141-147) - K2 of the exact two-phase key-frame graph, where the
 * warped feature must be materialised for the embedding / Nq convolutions:
 * out = w1*src0 + w2*cur, (w1,w2) = softmax over logits[n,0|1]; bypass[n] != 0 keeps cur.  NCHW f32. */
LSFA_API int lsfa_blend_logits_f32(const float* src0, const float* cur, const float* logits,
                                   const uint8_t* bypass, float* out, int N, int C, int H, int W,
                                   void* stream);

/* a15 - ChooseFeat (operator_py/choose_feat.py:23-31) with the flag kept on the device:
 * out[n] = eq_flag[n] ? conv_feat[n] : conv_feat_prop[n]; per_frame = C*H*W elements. */
LSFA_API int lsfa_choose_feat_f32(const float* conv_feat, const float* conv_feat_prop,
                                  const uint8_t* eq_flag, float* out, int N, long long per_frame,
                                  void* stream);

/* Upstream of the path (SURVEY.md 8f rank 3): coviar's accumulated MV field and residual for N GOPs at
 * once - external/data_loader_py2/coviar_data_loader.c:71-177 (create_and_load_mv_residual, accumulate=1)
 * with the identity initialisation of :318-328.
 * mvs: (N,T,M,6) int32 = per decoded P-frame t (1..T in decode order) up to M motion vectors, each
 *      {w, h, src_x, src_y, dst_x, dst_y} of FFmpeg's AVMotionVector in list order; counts (N,T) = how
 *      many are valid.  mv_out (N,height,width,2) int32 = what coviar_py2.load(.., 1, True) returns.
 * workspace: lsfa_mv_accumulate_workspace_bytes(N,height,width) bytes, no initialisation needed. */
LSFA_API size_t lsfa_mv_accumulate_workspace_bytes(int N, int height, int width);
LSFA_API int lsfa_mv_accumulate_i32(const int32_t* mvs, const int32_t* counts, int N, int T, int M, int height,
                                    int width, int32_t* mv_out, void* workspace, size_t workspace_bytes,
                                    void* stream);
/* The same with the algorithm pinned (ablation / tests): algo 0 auto, 1 the per-frame field form (owner map + gather, the
 * accumulated field crosses HBM every P-frame), 2 the cell-index back-trace (a chain of T look-ups per pixel through a
 * per-8x8-cell index; the field is written once; workspace lsfa_mv_accumulate_trace_workspace_bytes, N*T <= 65535).
 * lsfa_mv_accumulate_i32 = auto: the back-trace whenever it fits.  lsfa_mv_accumulate_workspace_bytes covers both. */
LSFA_API size_t lsfa_mv_accumulate_trace_workspace_bytes(int N, int T, int height, int width);
LSFA_API int lsfa_mv_accumulate_algo_i32(const int32_t* mvs, const int32_t* counts, int N, int T, int M, int height,
                                         int width, int32_t* mv_out, void* workspace, size_t workspace_bytes, int algo,
                                         void* stream);
/* residual of coviar_data_loader.c:141-175: res = cur - iframe[(x,y) - mv]; frames (N,height,width,3) uint8
 * BGR, mv the accumulated field above, res (N,height,width,3) int32. */
LSFA_API int lsfa_coviar_residual_u8(const uint8_t* iframe, const uint8_t* cur, const int32_t* mv, int32_t* res,
                                     int N, int height, int width, void* stream);

/* ---- backward of a7 / a8 (SURVEY.md 8f rank 4; get_train_symbol SYM:305-307,319-321) ---------------
 * MXNet BilinearSamplerBackward (src/operator/bilinear_sampler.cc) and GridGenerator Backward, kWarp
 * (src/operator/grid_generator-inl.h).  req_* follow OpReqType; kNullOp (or a NULL pointer) skips that
 * gradient - MXNet itself insists on both or neither, which is accepted here as a special case.
 *
 * a8 backward: data (N,C,Hi,Wi), grid (N,2,Ho,Wo), out_grad (N,C,Ho,Wo) ->
 *              grad_data (N,C,Hi,Wi), grad_grid (N,2,Ho,Wo); float32 NCHW.
 * workspace (optional, lsfa_bilinear_sampler_backward_workspace_bytes, 16-byte aligned, no initialisation
 * needed) enables the plane-resident gather kernel (deterministic grad_data, 3 launches); without it, or
 * for planes it cannot hold, the scatter kernel with global atomics runs (1 launch).
 * kernel: 0 auto, 1 scatter, 2 gather (LSFA_E_UNSUPPORTED if it cannot serve the arguments). */
LSFA_API size_t lsfa_bilinear_sampler_backward_workspace_bytes(int N, int C, int Hi, int Wi, int Ho, int Wo);
LSFA_API int lsfa_bilinear_sampler_backward_f32(const float* data, const float* grid, const float* out_grad,
                                                float* grad_data, float* grad_grid, int N, int C, int Hi, int Wi,
                                                int Ho, int Wo, int req_data, int req_grid, void* workspace,
                                                size_t workspace_bytes, int kernel, void* stream);
LSFA_API int lsfa_bilinear_sampler_backward_num_launches(int N, int C, int Hi, int Wi, int Ho, int Wo, int req_data,
                                                         int req_grid, size_t workspace_bytes, int kernel);
/* a7 backward: grad_flow = grad_grid / [(W-1)/2, (H-1)/2]; (N,2,H,W) float32. */
LSFA_API int lsfa_grid_generator_warp_backward_f32(const float* grad_grid, float* grad_flow, int N, int H, int W,
                                                   int req, void* stream);
/* a7+a8 backward in one pass: gradients of BilinearSampler(key, GridGenerator(flow, 'warp')) with respect
 * to key (N,C,H,W) and flow (N,2,H,W) (SYM:306-307: both; SYM:320-321: key only). */
LSFA_API int lsfa_warp_backward_f32(const float* key, const float* flow, const float* out_grad, float* grad_key,
                                    float* grad_flow, int N, int C, int H, int W, int req_key, int req_flow,
                                    void* workspace, size_t workspace_bytes, int kernel, void* stream);

/* ---- SURVEY.md 8f rank 2: the embedding / quality networks of the key-frame aggregation on tensor cores ----
 * Hand-written sm_100a implicit-GEMM convolutions (tcgen05.mma, fp32 accumulators in tensor memory, operands by
 * TMA tensor copies; lsfa_b200/csrc/conv_gemm_tc.cu).  Stated-tolerance variant: bf16 operands, fp32 accumulate
 * (the reference runs these convolutions in fp32 on cuDNN).  Activations are channels-last bf16 (NB,H,W,C);
 * The kernel pairs image b with image b + ceil(NB/2) on one weight tile (the reference always convolves Concat_0 of
 * two N-batches, SYM:95,133); lsfa_conv_bf16_nhwc also takes an odd NB (one image is then computed twice), the two
 * fused entry points need their 2N images.  Cin % 64 == 0, Cout % 256 == 0.
 *
 * weights: lsfa_pack_conv_weight_bf16 turns MXNet's (Cout,Cin,k,k) float32 into (Cout, k*k*Cin) bf16 (once per
 * parameter set).  bias stays float32. */
LSFA_API int lsfa_pack_conv_weight_bf16(const float* w, void* w_packed, int Cout, int Cin, int ksize, void* stream);
/* mx.sym.Convolution(kernel=(k,k), pad=(k/2,k/2), stride 1, no_bias=False) [+ Activation('relu')]: out (NB,H,W,Cout) bf16 */
LSFA_API int lsfa_conv_bf16_nhwc(const void* x, const void* w_packed, const float* bias, void* out, int NB, int H, int W,
                                 int Cin, int Cout, int ksize, int relu, void* stream);
/* get_embednet (SYM:118-130) + compute_weight (SYM:111-116) of Fgfa_net (SYM:132-139):
 * x = Concat_0(conv_feat, warp_feat) (2N,H,W,C) bf16 -> logits (N,2,H,W) f32, [n,0] = <e_warp^,e_cur^>, [n,1] = <e_cur^,e_cur^>
 * (the layout lsfa_blend_logits_f32 / LSFA_W_LOGITS consume).  em_conv3's 2048-channel output is reduced in the
 * GEMM epilogue and never written.  w1 (C1,C) 1x1, w2 (C2, 9*C1) 3x3, w3 (E, C2) 1x1, packed bf16.
 * workspace: lsfa_embed_cosine_logits_workspace_bytes, 256-byte aligned, no initialisation needed. */
LSFA_API size_t lsfa_embed_cosine_logits_workspace_bytes(int N, int H, int W, int C1, int C2, int E);
LSFA_API int lsfa_embed_cosine_logits_bf16_nhwc(const void* x, const void* w1, const float* b1, const void* w2,
                                                const float* b2, const void* w3, const float* b3, float* logits,
                                                int N, int H, int W, int C, int C1, int C2, int E, void* workspace,
                                                size_t workspace_bytes, void* stream);
/* the convolutions of Nq_net (SYM:95-101): x = Concat_0(warp_feat, conv_feat) (2N,H,W,C) bf16 -> logits (N,2,H,W) f32,
 * [n,0] = quality of the warped feature, [n,1] of the current one.  w1 = Nq_conv1 (256, 9*C) packed bf16; the
 * 256->16->1 tail (w2 (16,256), b2 (16), w3 (16), b3 (1), float32 device arrays) runs in the GEMM epilogue. */
LSFA_API int lsfa_nq_logits_bf16_nhwc(const void* x, const void* w1, const float* b1, const float* w2, const float* b2,
                                      const float* w3, const float* b3, float* logits, int N, int H, int W, int C,
                                      void* stream);

/* ---- backward of the fused operator's tails (SURVEY.md 8f rank 4; get_train_symbol SYM:306-338) -------------
 * Gradients of  out = wc*cur + ww*( BilinearSampler(key, GridGenerator(flow)) * scale_map + rnet_conv0(res) ),
 * (ww,wc) by weight_mode (NONE | ADD | MEAN | LOGITS = 2-way softmax | COSINE = softmax of the cosine logits), bypass
 * frames: out = cur, with respect to every
 * differentiable input, from d/d(out).  `fwd` is the forward's argument block (layout NCHW float32; `out` is not read
 * and may be any non-NULL pointer); each gradient has an OpReqType (NULL pointer or LSFA_REQ_NULL skips it).
 *   grad_key   (N,C,H,W)   needs private keys (key_index NULL) and key planes of the output's size
 *   grad_flow  (N,2,H,W)   LSFA_FLOW_PREPOOLED (flow in feature cells) or LSFA_FLOW_GRID (then it is d/d(grid));
 *                          raw motion vectors are integer data and get no gradient (SYM:319-321: the MV is data)
 *   grad_scale, grad_cur (N,C,H,W); grad_logits (N,2,H,W); grad_res (N,3,H,W); grad_rnet_w (C,3), grad_rnet_b (C)
 *   grad_emb_warp, grad_emb_cur (N,E,H,W)   LSFA_W_COSINE only (one req_emb for both; a NULL pointer skips one).  The
 *                          backward recomputes the cosine logits as the forward computes them with its full workspace
 *                          (with force_generic == 1: as the LDG pre-pass does), runs the LOGITS-mode backward on them
 *                          and then lsfa_cosine_logits_backward_f32_nchw.  grad_logits is not an output in this mode.
 * One pass over the feature streams (agg_tail_backward_kernel) + the a7/a8 gather backward for key/flow; every
 * reduction is summed in a fixed order (deterministic).  Bypass frames get zero embedding gradients (req = write) or
 * leave them untouched (req = add).  workspace: the _workspace_bytes query, 256-byte aligned.
 * struct_bytes may also be the size of the struct before the embedding fields, offsetof(LsfaAggGrads, grad_emb_warp):
 * those fields then read as NULL. */
typedef struct LsfaAggGrads {
  int32_t struct_bytes;        /* = sizeof(LsfaAggGrads) */
  const float* out_grad;       /* (N,C,H,W) */
  float* grad_key;    int32_t req_key;
  float* grad_flow;   int32_t req_flow;
  float* grad_scale;  int32_t req_scale;
  float* grad_cur;    int32_t req_cur;
  float* grad_logits; int32_t req_logits;
  float* grad_res;    int32_t req_res;
  float* grad_rnet_w; float* grad_rnet_b; int32_t req_rnet;
  void*  workspace;   size_t workspace_bytes;
  float* grad_emb_warp; float* grad_emb_cur; int32_t req_emb;
} LsfaAggGrads;
LSFA_API size_t lsfa_warp_scale_aggregate_backward_workspace_bytes(const LsfaAggArgs* fwd, const LsfaAggGrads* grads);
LSFA_API int    lsfa_warp_scale_aggregate_backward_f32_nchw(const LsfaAggArgs* fwd, const LsfaAggGrads* grads, void* stream);

/* layout helpers for the harness: NCHW f32 <-> NHWC {f32,bf16} */
LSFA_API int lsfa_nchw_to_nhwc(const float* src, void* dst, int N, int C, int H, int W, int dst_layout,
                      void* stream);
LSFA_API int lsfa_nhwc_to_nchw(const void* src, float* dst, int N, int C, int H, int W, int src_layout,
                      void* stream);

/* ---- record / replay (BASELINE configs[0]: the reference's batch-1 mode pays a launch per operator and frame) ----
 * Every entry point above only enqueues on the caller's stream - no allocation, no synchronisation, no host read-back -
 * so a sequence of calls can be captured into a CUDA graph and replayed with one launch.  These four wrap the CUDA
 * calls for callers that do not link the runtime themselves (MXNet's Python side: core/tester.py:138-145 issues the
 * operators of a frame one by one).  The captured calls' buffers (arguments, workspace) must stay alive and in place
 * for the lifetime of the graph; their CONTENTS may change between replays (new frame, same shapes).
 *   lsfa_graph_begin(stream)            cudaStreamBeginCapture (thread-local mode)
 *   ... any lsfa_* calls on `stream` ...
 *   lsfa_graph_end(stream, &g)          cudaStreamEndCapture + cudaGraphInstantiate -> opaque handle
 *   lsfa_graph_launch(g, stream)        cudaGraphLaunch        lsfa_graph_destroy(g)
 * An error between begin and end invalidates the capture: lsfa_graph_end then returns LSFA_E_CUDA and *graph = NULL. */
LSFA_API int lsfa_graph_begin(void* stream);
LSFA_API int lsfa_graph_end(void* stream, void** graph);
LSFA_API int lsfa_graph_launch(void* graph, void* stream);
LSFA_API int lsfa_graph_destroy(void* graph);

#ifdef __cplusplus
}
#endif
#endif /* LSFA_OPS_H_ */
