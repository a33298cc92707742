// extern "C" entry points declared in include/lsfa_ops.h: argument validation, tiling
// decisions and kernel launches.  No allocation, no synchronisation, no global mutable
// state; errors are reported through a thread-local message like MXGetLastError().
#include <cmath>
#include <cstdarg>
#include <cstddef>
#include <cstdio>
#include <cstring>

#include <new>

#include "lsfa_device.cuh"
#include "conv_gemm_tc.h"
#include "aggregate_backward.h"

namespace lsfa {
// aggregate_nchw.cu
bool plan_plane_kernel(AggParams& P, size_t* smem_out);
bool plan_tma_kernel(AggParams& P, size_t* smem_out);
bool plan_tma2_kernel(AggParams& P, size_t* smem_out, bool forced);
cudaError_t launch_agg_nchw_tma2(const AggParams& P, size_t smem, cudaStream_t st);
cudaError_t launch_agg_nchw_tma(const AggParams& P, size_t smem, cudaStream_t st);
cudaError_t launch_agg_nchw_plane(const AggParams& P, size_t smem, cudaStream_t st);
cudaError_t launch_agg_nchw_generic(const AggParams& P, cudaStream_t st);
cudaError_t launch_cosine_logits_nchw(const float* ew, const float* ec, float* logits, int N, int E,
                                      int HW, cudaStream_t st);
// cosine_nchw.cu
size_t cosine_tma_workspace_bytes(int N, int E, int HW);
cudaError_t launch_cosine_logits_nchw_tma(const float* ew, const float* ec, float* logits, int N, int E, int HW,
                                          void* scratch, size_t scratch_bytes, cudaStream_t st);
size_t cosine_backward_workspace_bytes(int N, int E, int HW);
cudaError_t launch_cosine_backward_nchw(const float* ew, const float* ec, const float* gl, const unsigned char* bypass, float* gw,
                                        float* gc, int add_w, int add_c, int N, int E, int HW, void* workspace,
                                        size_t workspace_bytes, bool tma_sums, int kernel, cudaStream_t st);
// aggregate_nhwc.cu
cudaError_t launch_agg_nhwc(const AggParams& P, bool bf16, int kernel, cudaStream_t st);
cudaError_t launch_cosine_logits_nhwc(const void* ew, const void* ec, float* logits, int N, int E,
                                      int HW, bool bf16, cudaStream_t st);
// prep_ops.cu
cudaError_t launch_mv_pool(const void* mv, bool is_i32, float* flow, int N, int h, int w, int H, int W,
                           double scale, int mode, cudaStream_t st);
cudaError_t launch_res_pool(const void* res, bool is_i32, float* out, int N, int h, int w, int H, int W,
                            const double* means, double pixel_scale, int mode, cudaStream_t st);
cudaError_t launch_res_coviar_pool(const int* res, float* out, int N, int h, int w, int oh, int ow, int H, int W,
                                   double im_scale, int hflip, const double* means, double pixel_scale, int mode,
                                   cudaStream_t st);
cudaError_t launch_mv_prepare(const int* in, float* out, int N, int h, int w, int oh, int ow,
                              double im_scale, int negate, int hflip, cudaStream_t st);
cudaError_t launch_grid_generator(const float* flow, float* grid, int N, int H, int W, float half_w,
                                  float half_h, cudaStream_t st);
cudaError_t launch_sampler_coords(const float* fg, int is_grid, int* x0, int* y0, float* wx, float* wy,
                                  int N, int H, int W, float half_w, float half_h, float wk_m1,
                                  float hk_m1, cudaStream_t st);
cudaError_t launch_nchw_to_nhwc(const float* src, void* dst, int N, int C, int HW, bool bf16, cudaStream_t st);
cudaError_t launch_nhwc_to_nchw(const void* src, float* dst, int N, int C, int HW, bool bf16, cudaStream_t st);
cudaError_t launch_unfused_chain(const float* key, const float* flow, const float* scale_map,
                                 const float* cur, const float* logits, float* out, float* tmp, int N,
                                 int C, int H, int W, float half_w, float half_h, cudaStream_t st);
int unfused_chain_launches();
cudaError_t launch_choose_feat(const float* a, const float* b, const unsigned char* flag, float* o,
                               long long per_frame, long long total, cudaStream_t st);
cudaError_t launch_blend_logits(const float* src0, const float* cur, const float* logits, const unsigned char* bypass,
                                float* out, int N, int C, int HW, cudaStream_t st);
// coviar_accumulate.cu
cudaError_t launch_mv_accumulate(const int* mvs, const int* counts, int N, int T, int M, int height, int width,
                                 int* mv_out, void* workspace, size_t workspace_bytes, int algo, cudaStream_t st);
size_t mvacc_trace_workspace_bytes(int N, int T, int height, int width);
cudaError_t launch_coviar_residual(const unsigned char* iframe, const unsigned char* cur, const int* mv, int* res, int N,
                                   int height, int width, cudaStream_t st);
// sampler_backward.cu
size_t bwd_workspace_bytes(int N, int HWk, int HW);
cudaError_t launch_sampler_backward(const float* data, const float* coords, int coords_is_flow, const float* og,
                                    float* gdata, float* ggrid, int N, int C, int Hi, int Wi, int Ho, int Wo,
                                    int add_data, int add_grid, float half_w, float half_h, void* workspace,
                                    size_t workspace_bytes, int kernel, cudaStream_t st);
int sampler_backward_num_launches(int N, int C, int Hi, int Wi, int Ho, int Wo, bool want_data, bool ws_ok, int kernel);
cudaError_t launch_grid_generator_backward(const float* g, float* o, int N, int H, int W, float half_w, float half_h,
                                           int add, cudaStream_t st);
}  // namespace lsfa

namespace {

thread_local char g_err[512] = "";

int fail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}

}  // namespace

namespace lsfa {
// for the other translation units that report through lsfa_last_error() (host_pipeline.cu)
int set_error(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}
}  // namespace lsfa

namespace {

int cuda_result(cudaError_t e, const char* what) {
  if (e == cudaSuccess) return LSFA_OK;
  return fail(LSFA_E_CUDA, "%s: %s", what, cudaGetErrorString(e));
}

inline cudaStream_t as_stream(void* s) { return static_cast<cudaStream_t>(s); }

// MXNet evaluates (DType(dim) - 1.0) / 2.0 in double and stores it as a float32 scalar.
inline float half_extent(int dim) { return (float)(((double)(float)dim - 1.0) / 2.0); }

inline int ceil16(int v) { return (v + 15) / 16; }

bool valid_req(int req) { return req >= LSFA_REQ_NULL && req <= LSFA_REQ_ADD; }

// Validate an LsfaAggArgs and translate it; returns LSFA_OK or an error code.
int build_params(const LsfaAggArgs* a, lsfa::AggParams& P) {
  if (!a) return fail(LSFA_E_BADARG, "args is NULL");
  if (a->struct_bytes != (int32_t)sizeof(LsfaAggArgs))
    return fail(LSFA_E_BADARG, "args->struct_bytes=%d, this library expects %zu (ABI %d)",
                a->struct_bytes, sizeof(LsfaAggArgs), LSFA_ABI_VERSION);
  if (a->layout < LSFA_LAYOUT_NCHW_F32 || a->layout > LSFA_LAYOUT_NHWC_BF16)
    return fail(LSFA_E_BADARG, "unknown layout %d", a->layout);
  if (a->N <= 0 || a->C <= 0 || a->H <= 0 || a->W <= 0)
    return fail(LSFA_E_SHAPE, "non-positive dims N=%d C=%d H=%d W=%d", a->N, a->C, a->H, a->W);
  if (!valid_req(a->req)) return fail(LSFA_E_BADARG, "unknown req %d", a->req);
  const int Hk = a->key_h > 0 ? a->key_h : a->H, Wk = a->key_w > 0 ? a->key_w : a->W;
  if ((a->key_h > 0) != (a->key_w > 0)) return fail(LSFA_E_SHAPE, "key_h/key_w must both be set or both 0");
  if ((long long)a->H * a->W >= (1LL << 24) || (long long)Hk * Wk >= (1LL << 24))
    return fail(LSFA_E_SHAPE, "planes of 2^24 pixels or more are not supported");
  if (!a->key || !a->flow || !a->out) return fail(LSFA_E_BADARG, "key, flow and out are required");
  if (a->flow_kind < LSFA_FLOW_PREPOOLED || a->flow_kind > LSFA_FLOW_COVIAR_I32)
    return fail(LSFA_E_BADARG, "unknown flow_kind %d", a->flow_kind);
  if (a->flow_kind == LSFA_FLOW_COVIAR_I32) {
    if (a->mv_src_h <= 0 || a->mv_src_w <= 0) return fail(LSFA_E_SHAPE, "LSFA_FLOW_COVIAR_I32 needs mv_src_h, mv_src_w > 0");
    if (!(a->im_scale > 0.0)) return fail(LSFA_E_BADARG, "im_scale must be > 0");
    const long eh = a->im_scale == 1.0 ? a->mv_src_h : lrint((double)a->mv_src_h * a->im_scale);   // cvRound
    const long ew = a->im_scale == 1.0 ? a->mv_src_w : lrint((double)a->mv_src_w * a->im_scale);
    if (a->mv_h != eh || a->mv_w != ew)
      return fail(LSFA_E_SHAPE, "coviar %dx%d at im_scale %g resizes to %ldx%ld, but mv_h,mv_w = %d,%d", a->mv_src_h,
                  a->mv_src_w, a->im_scale, eh, ew, a->mv_h, a->mv_w);
  }
  if (a->flow_kind == LSFA_FLOW_RAW_I32 || a->flow_kind == LSFA_FLOW_RAW_F32 || a->flow_kind == LSFA_FLOW_COVIAR_I32) {
    if (a->mv_h <= 0 || a->mv_w <= 0) return fail(LSFA_E_SHAPE, "raw MV needs mv_h, mv_w > 0");
    if (ceil16(a->mv_h) != a->H || ceil16(a->mv_w) != a->W)
      return fail(LSFA_E_SHAPE, "raw MV %dx%d pools to %dx%d, but H,W = %d,%d", a->mv_h, a->mv_w,
                  ceil16(a->mv_h), ceil16(a->mv_w), a->H, a->W);
    if (a->pool_mode != LSFA_POOL_CENTRE2X2 && a->pool_mode != LSFA_POOL_AVG16)
      return fail(LSFA_E_BADARG, "unknown pool_mode %d", a->pool_mode);
    if (!(a->im_scale > 0.0)) return fail(LSFA_E_BADARG, "im_scale must be > 0");
  }
  if (a->weight_mode < LSFA_W_NONE || a->weight_mode > LSFA_W_COSINE)
    return fail(LSFA_E_BADARG, "unknown weight_mode %d", a->weight_mode);
  if (a->weight_mode != LSFA_W_NONE && !a->cur) return fail(LSFA_E_BADARG, "cur is required for weight_mode %d", a->weight_mode);
  if (a->weight_mode == LSFA_W_LOGITS && !a->logits) return fail(LSFA_E_BADARG, "logits is required for LSFA_W_LOGITS");
  if (a->weight_mode == LSFA_W_COSINE) {
    if (!a->emb_warp || !a->emb_cur) return fail(LSFA_E_BADARG, "emb_warp and emb_cur are required for LSFA_W_COSINE");
    if (a->E <= 0) return fail(LSFA_E_SHAPE, "E must be > 0 for LSFA_W_COSINE");
  }
  if (a->bypass && a->weight_mode == LSFA_W_NONE)
    return fail(LSFA_E_BADARG, "bypass needs cur (weight_mode != NONE)");
  if (a->res && (!a->rnet_w || !a->rnet_b)) return fail(LSFA_E_BADARG, "res needs rnet_w and rnet_b");
  if (a->key_index && a->num_keys <= 0) return fail(LSFA_E_BADARG, "key_index needs num_keys > 0");
  if (a->layout != LSFA_LAYOUT_NCHW_F32) {
    const int lanes = a->layout == LSFA_LAYOUT_NHWC_BF16 ? 8 : 4;
    if (a->C % lanes) return fail(LSFA_E_ALIGN, "NHWC layout needs C %% %d == 0 (C=%d)", lanes, a->C);
    if (a->weight_mode == LSFA_W_COSINE && a->E % lanes)
      return fail(LSFA_E_ALIGN, "NHWC layout needs E %% %d == 0 (E=%d)", lanes, a->E);
    const void* ptrs[] = {a->key, a->scale_map, a->cur, a->out, a->emb_warp, a->emb_cur};
    for (const void* p : ptrs)
      if (p && (reinterpret_cast<uintptr_t>(p) % 16))
        return fail(LSFA_E_ALIGN, "NHWC tensors must be 16-byte aligned");
  }

  memset(&P, 0, sizeof(P));
  P.N = a->N; P.C = a->C; P.H = a->H; P.W = a->W; P.HW = a->H * a->W;
  P.Hk = Hk; P.Wk = Wk; P.HWk = Hk * Wk;
  P.key = a->key; P.key_index = a->key_index;
  P.num_keys = a->num_keys > 0 ? a->num_keys : a->N;
  P.flow_kind = a->flow_kind; P.flow = a->flow;
  P.mv_h = a->mv_h; P.mv_w = a->mv_w;
  P.mv_scale = a->im_scale * (1.0 / 16.0);      // image.py:224: scale = im_scale * rcnn_scale
  P.pool_mode = a->pool_mode;
  P.src_h = a->mv_src_h; P.src_w = a->mv_src_w;
  P.inv_scale = a->im_scale > 0.0 ? 1.0 / a->im_scale : 1.0;
  P.mv_negate = a->mv_negate; P.mv_hflip = a->mv_hflip; P.mv_identity = a->im_scale == 1.0;
  P.scale = a->scale_map; P.res = a->res; P.rnet_w = a->rnet_w; P.rnet_b = a->rnet_b;
  P.cur = a->cur; P.mode = a->weight_mode; P.logits = a->logits;
  P.emb_warp = a->emb_warp; P.emb_cur = a->emb_cur; P.E = a->E;
  P.bypass = a->bypass; P.out = a->out; P.req_add = a->req == LSFA_REQ_ADD;
  P.half_w = half_extent(a->W); P.half_h = half_extent(a->H);
  P.wk_m1 = (float)(Wk - 1); P.hk_m1 = (float)(Hk - 1);
  return LSFA_OK;
}

// Workspace layout (NCHW only): [cosine logits (N,2,H,W) f32, COSINE mode only][claim counters][records]
size_t cosine_ws_bytes(const LsfaAggArgs* a) {
  if (!a || a->weight_mode != LSFA_W_COSINE || a->layout != LSFA_LAYOUT_NCHW_F32) return 0;
  if (a->N <= 0 || a->H <= 0 || a->W <= 0) return 0;
  return (size_t)a->N * 2 * a->H * a->W * sizeof(float);
}
size_t cosine_partials_ws_bytes(const LsfaAggArgs* a) {   // partial sums of the all-TMA cosine pre-pass (optional)
  if (cosine_ws_bytes(a) == 0 || a->E <= 0) return 0;
  return (lsfa::cosine_tma_workspace_bytes(a->N, a->E, a->H * a->W) + 15) / 16 * 16;
}
size_t records_ws_bytes(const LsfaAggArgs* a) {   // packed sampling records of the pre-pass: 32 B per output pixel
  if (!a || a->layout != LSFA_LAYOUT_NCHW_F32 || a->N <= 0 || a->H <= 0 || a->W <= 0) return 0;
  return (size_t)a->N * a->H * a->W * 32;
}
constexpr size_t kNhwcWorkspaceBytes = 64;   // channels-last: one claim counter (padded)

size_t sched_ws_bytes(const LsfaAggArgs* a) {
  if (!a || a->layout != LSFA_LAYOUT_NCHW_F32 || a->N <= 0 || a->H <= 0 || a->W <= 0) return 0;
  const size_t parts = ((size_t)a->H * a->W + 4319) / 4320;      // pixel parts of the all-TMA kernel (9 x 480)
  return ((size_t)a->N * parts * sizeof(unsigned) * 3 + 15) / 16 * 16;   // claim counters + 2 row-range words per part
}

// cosine logits (N,2,H,W) of NCHW embeddings: the all-TMA pre-pass where it serves and `scratch` holds its partial sums
// (unless tma is false), else the LDG kernel.  The fused forward and the fused backward both compute them here.
cudaError_t cosine_logits_nchw(const float* ew, const float* ec, float* lg, int N, int E, int HW, void* scratch,
                               size_t scratch_bytes, bool tma, cudaStream_t st) {
  cudaError_t ce = cudaErrorNotSupported;
  if (tma) ce = lsfa::launch_cosine_logits_nchw_tma(ew, ec, lg, N, E, HW, scratch, scratch_bytes, st);
  if (ce == cudaErrorNotSupported) ce = lsfa::launch_cosine_logits_nchw(ew, ec, lg, N, E, HW, st);
  return ce;
}
int run_aggregate(const LsfaAggArgs* a, void* stream) {
  lsfa::AggParams P;
  int rc = build_params(a, P);
  if (rc != LSFA_OK) return rc;
  if (a->req == LSFA_REQ_NULL) return LSFA_OK;
  cudaStream_t st = as_stream(stream);
  if (a->layout == LSFA_LAYOUT_NCHW_F32) {
    if (a->weight_mode == LSFA_W_COSINE) {
      // NCHW embeddings are channel-planar: the per-pixel cosine needs its own pass over
      // them (each byte still read once); its (N,2,H,W) result feeds the fused kernel.
      const size_t need = cosine_ws_bytes(a);
      if (!a->workspace || a->workspace_bytes < need)
        return fail(LSFA_E_BADARG, "LSFA_W_COSINE in NCHW needs a workspace of %zu bytes", need);
      if (reinterpret_cast<uintptr_t>(a->workspace) % 4) return fail(LSFA_E_ALIGN, "workspace must be 4-byte aligned");
      float* lg = static_cast<float*>(a->workspace);
      // with the full workspace: all-TMA pre-pass (deterministic partial sums); else the LDG kernel
      const size_t lg_b = (need + 15) / 16 * 16, part_b = cosine_partials_ws_bytes(a);
      const bool tma = part_b && a->workspace_bytes >= lg_b + part_b && (reinterpret_cast<uintptr_t>(a->workspace) % 16) == 0 &&
                       a->force_generic != 1;
      rc = cuda_result(cosine_logits_nchw(static_cast<const float*>(a->emb_warp), static_cast<const float*>(a->emb_cur), lg, a->N,
                                          a->E, P.HW, static_cast<char*>(a->workspace) + lg_b, part_b, tma, st),
                       "cosine_logits_nchw launch");
      if (rc != LSFA_OK) return rc;
      P.logits = lg;
    }
    // optional scratch for dynamic work claiming (all-TMA kernel); without it the split is static
    const size_t cos_b = (cosine_ws_bytes(a) + 15) / 16 * 16 + cosine_partials_ws_bytes(a);
    const size_t ws_need = cos_b + sched_ws_bytes(a) + records_ws_bytes(a);
    if (a->workspace && a->workspace_bytes >= ws_need && (reinterpret_cast<uintptr_t>(a->workspace) % 16) == 0) {
      char* ws = static_cast<char*>(a->workspace);
      P.sched = reinterpret_cast<unsigned*>(ws + cos_b);
      P.records = reinterpret_cast<const uint4*>(ws + cos_b + sched_ws_bytes(a));
    }
    size_t smem = 0;
    // kernel choice: 0 auto (all-TMA, then plane-resident LDG/STG, then generic); the other
    // values pin one kernel for tests and ablations
    // The 2-CTA cluster form (multicast key load) is opt-in: measured on 1024x68x120 it reaches 0.65 of the
    // HBM peak against 0.81 for the single-CTA kernel with two pixel parts - with only 3 stages of 67 KB the
    // cross-CTA hand-shake per refill (peer_free -> claim -> desc_ready) leaves the pair latency-bound.
    if (a->force_generic == 4 && lsfa::plan_tma2_kernel(P, &smem, true))
      return cuda_result(lsfa::launch_agg_nchw_tma2(P, smem, st), "agg_nchw_tma2 launch");
    if (a->force_generic == 4) return fail(LSFA_E_UNSUPPORTED, "the 2-CTA cluster kernel cannot serve these arguments");
    if ((a->force_generic == 0 || a->force_generic == 3) && lsfa::plan_tma_kernel(P, &smem))
      return cuda_result(lsfa::launch_agg_nchw_tma(P, smem, st), "agg_nchw_tma launch");
    if (a->force_generic == 3) return fail(LSFA_E_UNSUPPORTED, "the all-TMA kernel cannot serve these arguments");
    if (a->force_generic != 1 && lsfa::plan_plane_kernel(P, &smem))
      return cuda_result(lsfa::launch_agg_nchw_plane(P, smem, st), "agg_nchw_plane launch");
    return cuda_result(lsfa::launch_agg_nchw_generic(P, st), "agg_nchw_generic launch");
  }
  // channels-last: force_generic 0 = auto, 1 = LDG/STG tile kernel, 3 = all-TMA gather-by-bulk-copy or fail,
  // 5 = window-resident all-TMA (tensor maps) or fail.
  // An optional 64-byte workspace holds the claim counter of the all-TMA kernels (NULL = static stride).
  if (a->force_generic != 0 && a->force_generic != 1 && a->force_generic != 3 && a->force_generic != 5)
    return fail(LSFA_E_BADARG, "force_generic %d is not defined for the channels-last layouts (0, 1, 3 or 5)", a->force_generic);
  if (a->workspace && a->workspace_bytes >= kNhwcWorkspaceBytes && (reinterpret_cast<uintptr_t>(a->workspace) % 4) == 0)
    P.sched = static_cast<unsigned*>(a->workspace);
  cudaError_t e = lsfa::launch_agg_nhwc(P, a->layout == LSFA_LAYOUT_NHWC_BF16, a->force_generic, st);
  if (e == cudaErrorNotSupported) {
    cudaGetLastError();
    return fail(LSFA_E_UNSUPPORTED, "the all-TMA channels-last kernel cannot serve these arguments");
  }
  return cuda_result(e, "agg_nhwc launch");
}

}  // namespace

extern "C" {

int lsfa_version(void) { return LSFA_ABI_VERSION; }

const char* lsfa_last_error(void) { return g_err; }

static int mv_pool_common(const void* mv, bool is_i32, float* flow, int N, int h, int w, double im_scale,
                          int mode, void* stream) {
  if (!mv || !flow) return fail(LSFA_E_BADARG, "mv and flow are required");
  if (N <= 0 || h <= 0 || w <= 0) return fail(LSFA_E_SHAPE, "non-positive dims N=%d h=%d w=%d", N, h, w);
  if (mode != LSFA_POOL_CENTRE2X2 && mode != LSFA_POOL_AVG16) return fail(LSFA_E_BADARG, "unknown pool mode %d", mode);
  if (!(im_scale > 0.0)) return fail(LSFA_E_BADARG, "im_scale must be > 0");
  return cuda_result(lsfa::launch_mv_pool(mv, is_i32, flow, N, h, w, ceil16(h), ceil16(w),
                                          im_scale * (1.0 / 16.0), mode, as_stream(stream)),
                     "mv_pool launch");
}
int lsfa_mv_pool_i32(const int32_t* mv, float* flow, int N, int h, int w, double im_scale, int mode, void* stream) {
  return mv_pool_common(mv, true, flow, N, h, w, im_scale, mode, stream);
}
int lsfa_mv_pool_f32(const float* mv, float* flow, int N, int h, int w, double im_scale, int mode, void* stream) {
  return mv_pool_common(mv, false, flow, N, h, w, im_scale, mode, stream);
}

static int res_pool_common(const void* res, bool is_i32, float* out, int N, int h, int w, const double* means,
                           double pixel_scale, int mode, void* stream) {
  if (!res || !out) return fail(LSFA_E_BADARG, "res and out are required");
  if (N <= 0 || h <= 0 || w <= 0) return fail(LSFA_E_SHAPE, "non-positive dims N=%d h=%d w=%d", N, h, w);
  if (mode != LSFA_POOL_CENTRE2X2 && mode != LSFA_POOL_AVG16) return fail(LSFA_E_BADARG, "unknown pool mode %d", mode);
  return cuda_result(lsfa::launch_res_pool(res, is_i32, out, N, h, w, ceil16(h), ceil16(w), means, pixel_scale,
                                           mode, as_stream(stream)),
                     "res_pool launch");
}
int lsfa_res_pool_i32(const int32_t* res, float* out, int N, int h, int w, const double* means,
                      double pixel_scale, int mode, void* stream) {
  return res_pool_common(res, true, out, N, h, w, means, pixel_scale, mode, stream);
}
int lsfa_res_pool_f32(const float* res, float* out, int N, int h, int w, const double* means,
                      double pixel_scale, int mode, void* stream) {
  return res_pool_common(res, false, out, N, h, w, means, pixel_scale, mode, stream);
}

int lsfa_res_coviar_pool_i32(const int32_t* res_coviar, float* out, int N, int h, int w, int oh, int ow, double im_scale,
                             int hflip, const double* means, double pixel_scale, int mode, void* stream) {
  if (!res_coviar || !out) return fail(LSFA_E_BADARG, "res_coviar and out are required");
  if (N <= 0 || h <= 0 || w <= 0 || oh <= 0 || ow <= 0) return fail(LSFA_E_SHAPE, "non-positive dims");
  if (mode != LSFA_POOL_CENTRE2X2 && mode != LSFA_POOL_AVG16) return fail(LSFA_E_BADARG, "unknown pool mode %d", mode);
  if (!(im_scale > 0.0)) return fail(LSFA_E_BADARG, "im_scale must be > 0");
  const long eh = im_scale == 1.0 ? h : lrint((double)h * im_scale), ew = im_scale == 1.0 ? w : lrint((double)w * im_scale);
  if (oh != eh || ow != ew)
    return fail(LSFA_E_SHAPE, "residual %dx%d at im_scale %g resizes to %ldx%ld, but oh,ow = %d,%d", h, w, im_scale, eh, ew, oh, ow);
  return cuda_result(lsfa::launch_res_coviar_pool(res_coviar, out, N, h, w, oh, ow, ceil16(oh), ceil16(ow), im_scale, hflip,
                                                  means, pixel_scale, mode, as_stream(stream)),
                     "res_coviar_pool launch");
}

int lsfa_mv_centre_rows_h2d(const void* mv_host, void* mv_dev, int N, int h, int w, size_t* bytes_out, void* stream) {
  if (!mv_host || !mv_dev) return fail(LSFA_E_BADARG, "mv_host and mv_dev are required");
  if (N <= 0 || h <= 0 || w <= 0) return fail(LSFA_E_SHAPE, "non-positive dims N=%d h=%d w=%d", N, h, w);
  const size_t row = (size_t)w * 8, frame = row * (size_t)h, pitch = 16 * row;
  const int pairs = (h - 7) / 16 + ((h - 7) % 16 >= 2 ? 1 : 0);     // blocks whose rows 16k+7 AND 16k+8 both exist
  const bool lone = h >= 8 && (h - 8) % 16 == 0;                      // a last block with row 16k+7 only
  size_t bytes = 0;
  cudaStream_t st = as_stream(stream);
  for (int n = 0; n < N; ++n) {
    const char* src = static_cast<const char*>(mv_host) + (size_t)n * frame + 7 * row;
    char* dst = static_cast<char*>(mv_dev) + (size_t)n * frame + 7 * row;
    if (pairs > 0) {
      cudaError_t e = cudaMemcpy2DAsync(dst, pitch, src, pitch, 2 * row, (size_t)pairs, cudaMemcpyHostToDevice, st);
      if (e != cudaSuccess) return cuda_result(e, "mv_centre_rows_h2d");
      bytes += 2 * row * (size_t)pairs;
    }
    if (lone) {
      const size_t off = (size_t)(h - 1 - 7) * row;
      cudaError_t e = cudaMemcpyAsync(dst + off, src + off, row, cudaMemcpyHostToDevice, st);
      if (e != cudaSuccess) return cuda_result(e, "mv_centre_rows_h2d");
      bytes += row;
    }
  }
  if (bytes_out) *bytes_out = bytes;
  return LSFA_OK;
}

int lsfa_mv_prepare_i32(const int32_t* mv_coviar, float* mv_out, int N, int h, int w, int oh, int ow,
                        double im_scale, int negate, int hflip, void* stream) {
  if (!mv_coviar || !mv_out) return fail(LSFA_E_BADARG, "mv_coviar and mv_out are required");
  if (N <= 0 || h <= 0 || w <= 0 || oh <= 0 || ow <= 0) return fail(LSFA_E_SHAPE, "non-positive dims");
  if (!(im_scale > 0.0)) return fail(LSFA_E_BADARG, "im_scale must be > 0");
  if (im_scale == 1.0 && (oh != h || ow != w)) return fail(LSFA_E_SHAPE, "im_scale 1 needs oh,ow == h,w");
  if (reinterpret_cast<uintptr_t>(mv_out) % 8) return fail(LSFA_E_ALIGN, "mv_out must be 8-byte aligned");
  return cuda_result(lsfa::launch_mv_prepare(mv_coviar, mv_out, N, h, w, oh, ow, im_scale, negate, hflip,
                                             as_stream(stream)),
                     "mv_prepare launch");
}

int lsfa_grid_generator_warp_f32(const float* flow, float* grid, int N, int H, int W, void* stream) {
  if (!flow || !grid) return fail(LSFA_E_BADARG, "flow and grid are required");
  if (N <= 0 || H <= 0 || W <= 0) return fail(LSFA_E_SHAPE, "non-positive dims N=%d H=%d W=%d", N, H, W);
  return cuda_result(lsfa::launch_grid_generator(flow, grid, N, H, W, half_extent(W), half_extent(H),
                                                 as_stream(stream)),
                     "grid_generator launch");
}

int lsfa_bilinear_sampler_f32(const float* data, const float* grid, float* out, int N, int C, int Hi, int Wi,
                              int Ho, int Wo, int req, void* stream) {
  LsfaAggArgs a;
  memset(&a, 0, sizeof(a));
  a.struct_bytes = (int32_t)sizeof(a);
  a.layout = LSFA_LAYOUT_NCHW_F32;
  a.N = N; a.C = C; a.H = Ho; a.W = Wo; a.key_h = Hi; a.key_w = Wi;
  a.key = data; a.flow_kind = LSFA_FLOW_GRID; a.flow = grid;
  a.weight_mode = LSFA_W_NONE; a.out = out; a.req = req;
  if (Hi <= 0 || Wi <= 0) return fail(LSFA_E_SHAPE, "non-positive input plane %dx%d", Hi, Wi);
  return run_aggregate(&a, stream);
}

int lsfa_sampler_coords_f32(const float* flow_or_grid, int is_grid, int32_t* x0, int32_t* y0, float* wx,
                            float* wy, int N, int H, int W, int Hi, int Wi, void* stream) {
  if (!flow_or_grid || !x0 || !y0 || !wx || !wy) return fail(LSFA_E_BADARG, "NULL pointer");
  if (N <= 0 || H <= 0 || W <= 0 || Hi <= 0 || Wi <= 0) return fail(LSFA_E_SHAPE, "non-positive dims");
  return cuda_result(lsfa::launch_sampler_coords(flow_or_grid, is_grid, x0, y0, wx, wy, N, H, W, half_extent(W),
                                                 half_extent(H), (float)(Wi - 1), (float)(Hi - 1),
                                                 as_stream(stream)),
                     "sampler_coords launch");
}

int lsfa_warp_scale_aggregate(const LsfaAggArgs* args, void* stream) { return run_aggregate(args, stream); }

int lsfa_warp_scale_aggregate_f32_nchw(const LsfaAggArgs* args, void* stream) {
  if (args && args->layout != LSFA_LAYOUT_NCHW_F32)
    return fail(LSFA_E_BADARG, "lsfa_warp_scale_aggregate_f32_nchw called with layout %d", args->layout);
  return run_aggregate(args, stream);
}

int lsfa_warp_scale_aggregate_bf16_nhwc(const LsfaAggArgs* args, void* stream) {
  if (args && args->layout != LSFA_LAYOUT_NHWC_BF16)
    return fail(LSFA_E_BADARG, "lsfa_warp_scale_aggregate_bf16_nhwc called with layout %d", args->layout);
  return run_aggregate(args, stream);
}

size_t lsfa_warp_scale_aggregate_workspace_bytes(const LsfaAggArgs* args) {
  if (args && (args->layout == LSFA_LAYOUT_NHWC_F32 || args->layout == LSFA_LAYOUT_NHWC_BF16)) return kNhwcWorkspaceBytes;
  return (cosine_ws_bytes(args) + 15) / 16 * 16 + cosine_partials_ws_bytes(args) + sched_ws_bytes(args) + records_ws_bytes(args);
}

int lsfa_warp_scale_aggregate_num_launches(const LsfaAggArgs* args) {
  if (!args || args->req == LSFA_REQ_NULL) return 0;
  if (args->layout != LSFA_LAYOUT_NCHW_F32) return 1;
  int n = 1;
  if (args->weight_mode == LSFA_W_COSINE) {                          // cosine-logit pre-pass (+ its finalize when all-TMA)
    ++n;
    const size_t full = lsfa_warp_scale_aggregate_workspace_bytes(args);
    if (cosine_partials_ws_bytes(args) && args->workspace && args->workspace_bytes >= full && args->force_generic != 1) ++n;
  }
  const size_t need = lsfa_warp_scale_aggregate_workspace_bytes(args);
  if (args->workspace && args->workspace_bytes >= need && args->force_generic != 1 && args->force_generic != 2) {
    // record pre-pass of the all-TMA kernel - except for small batches (N x pixel parts <= 8), which the kernel serves in
    // ONE cooperative launch: its own consumers build the records before a grid-wide barrier
    const long long parts = ((long long)args->H * args->W + 4319) / 4320;
    if (args->force_generic == 4 || (long long)args->N * parts > 8) ++n;
  }
  return n;
}

int lsfa_cosine_logits(const void* emb_warp, const void* emb_cur, float* logits, int N, int E, int H, int W,
                       int layout, void* stream) {
  if (!emb_warp || !emb_cur || !logits) return fail(LSFA_E_BADARG, "NULL pointer");
  if (N <= 0 || E <= 0 || H <= 0 || W <= 0) return fail(LSFA_E_SHAPE, "non-positive dims");
  if (layout == LSFA_LAYOUT_NCHW_F32)
    return cuda_result(lsfa::launch_cosine_logits_nchw(static_cast<const float*>(emb_warp),
                                                       static_cast<const float*>(emb_cur), logits, N, E, H * W,
                                                       as_stream(stream)),
                       "cosine_logits_nchw launch");
  if (layout != LSFA_LAYOUT_NHWC_F32 && layout != LSFA_LAYOUT_NHWC_BF16) return fail(LSFA_E_BADARG, "unknown layout %d", layout);
  const int lanes = layout == LSFA_LAYOUT_NHWC_BF16 ? 8 : 4;
  if (E % lanes) return fail(LSFA_E_ALIGN, "NHWC layout needs E %% %d == 0", lanes);
  if ((reinterpret_cast<uintptr_t>(emb_warp) % 16) || (reinterpret_cast<uintptr_t>(emb_cur) % 16))
    return fail(LSFA_E_ALIGN, "NHWC tensors must be 16-byte aligned");
  return cuda_result(lsfa::launch_cosine_logits_nhwc(emb_warp, emb_cur, logits, N, E, H * W,
                                                     layout == LSFA_LAYOUT_NHWC_BF16, as_stream(stream)),
                     "cosine_logits_nhwc launch");
}

size_t lsfa_cosine_logits_workspace_bytes(int N, int E, int H, int W, int layout) {
  if (layout != LSFA_LAYOUT_NCHW_F32 || N <= 0 || E <= 0 || H <= 0 || W <= 0) return 0;
  return lsfa::cosine_tma_workspace_bytes(N, E, H * W);
}

int lsfa_cosine_logits_ws(const void* emb_warp, const void* emb_cur, float* logits, int N, int E, int H, int W, int layout,
                          void* workspace, size_t workspace_bytes, void* stream) {
  if (layout == LSFA_LAYOUT_NCHW_F32 && emb_warp && emb_cur && logits && N > 0 && E > 0 && H > 0 && W > 0 && workspace) {
    cudaError_t e = lsfa::launch_cosine_logits_nchw_tma(static_cast<const float*>(emb_warp), static_cast<const float*>(emb_cur),
                                                        logits, N, E, H * W, workspace, workspace_bytes, as_stream(stream));
    if (e != cudaErrorNotSupported) return cuda_result(e, "cosine_logits_nchw_tma launch");
  }
  return lsfa_cosine_logits(emb_warp, emb_cur, logits, N, E, H, W, layout, stream);
}

size_t lsfa_cosine_logits_backward_workspace_bytes(int N, int E, int H, int W) {
  if (N <= 0 || E <= 0 || H <= 0 || W <= 0) return 0;
  return lsfa::cosine_backward_workspace_bytes(N, E, H * W);
}

static bool overlaps(const void* p, size_t pb, const void* q, size_t qb) {
  const uintptr_t a = reinterpret_cast<uintptr_t>(p), b = reinterpret_cast<uintptr_t>(q);
  return p && q && a < b + qb && b < a + pb;
}

int lsfa_cosine_logits_backward_f32_nchw(const float* emb_warp, const float* emb_cur, const float* grad_logits,
                                         float* grad_emb_warp, float* grad_emb_cur, int N, int E, int H, int W, int req_warp,
                                         int req_cur, void* workspace, size_t workspace_bytes, int kernel, void* stream) {
  if (!valid_req(req_warp) || !valid_req(req_cur)) return fail(LSFA_E_BADARG, "unknown req %d / %d", req_warp, req_cur);
  if (kernel < 0 || kernel > 2) return fail(LSFA_E_BADARG, "kernel must be 0 (auto), 1 (plain) or 2 (all-TMA)");
  if (N <= 0 || E <= 0 || H <= 0 || W <= 0) return fail(LSFA_E_SHAPE, "non-positive dims N=%d E=%d H=%d W=%d", N, E, H, W);
  if ((long long)H * W >= (1LL << 24)) return fail(LSFA_E_SHAPE, "planes of 2^24 pixels or more are not supported");
  if (N > 65535) return fail(LSFA_E_SHAPE, "N must be at most 65535");
  if (req_warp == LSFA_REQ_NULL) grad_emb_warp = nullptr;
  if (req_cur == LSFA_REQ_NULL) grad_emb_cur = nullptr;
  if (!grad_emb_warp && !grad_emb_cur) return LSFA_OK;                  // nothing requested
  if (!emb_warp || !emb_cur || !grad_logits) return fail(LSFA_E_BADARG, "emb_warp, emb_cur and grad_logits are required");
  const size_t eb = (size_t)N * E * H * W * sizeof(float), lb = (size_t)N * 2 * H * W * sizeof(float);
  for (const float* gp : {(const float*)grad_emb_warp, (const float*)grad_emb_cur})
    if (overlaps(gp, eb, emb_warp, eb) || overlaps(gp, eb, emb_cur, eb) || overlaps(gp, eb, grad_logits, lb))
      return fail(LSFA_E_BADARG, "the gradients must not overlap emb_warp, emb_cur or grad_logits");
  if (overlaps(grad_emb_warp, eb, grad_emb_cur, eb)) return fail(LSFA_E_BADARG, "grad_emb_warp and grad_emb_cur overlap");
  const size_t need = lsfa::cosine_backward_workspace_bytes(N, E, H * W);
  if (!workspace || workspace_bytes < need) return fail(LSFA_E_BADARG, "workspace too small: need %zu bytes", need);
  if (reinterpret_cast<uintptr_t>(workspace) % 16) return fail(LSFA_E_ALIGN, "workspace must be 16-byte aligned");
  cudaError_t e = lsfa::launch_cosine_backward_nchw(emb_warp, emb_cur, grad_logits, nullptr, grad_emb_warp, grad_emb_cur,
                                                    req_warp == LSFA_REQ_ADD, req_cur == LSFA_REQ_ADD, N, E, H * W, workspace,
                                                    workspace_bytes, true, kernel, as_stream(stream));
  if (e == cudaErrorNotSupported) {
    cudaGetLastError();
    return fail(LSFA_E_UNSUPPORTED, "the all-TMA kernel cannot serve these arguments (plane size, odd E or H*W, alignment)");
  }
  return cuda_result(e, "cosine backward launch");
}

int lsfa_unfused_chain_f32_nchw(const float* key, const float* flow, const float* scale_map, const float* cur,
                                const float* logits, float* out, float* tmp, int N, int C, int H, int W,
                                void* stream) {
  if (!key || !flow || !scale_map || !cur || !logits || !out || !tmp) return fail(LSFA_E_BADARG, "NULL pointer");
  if (N <= 0 || C < 4 || H <= 0 || W <= 0) return fail(LSFA_E_SHAPE, "need N,H,W > 0 and C >= 4");
  return cuda_result(lsfa::launch_unfused_chain(key, flow, scale_map, cur, logits, out, tmp, N, C, H, W,
                                                half_extent(W), half_extent(H), as_stream(stream)),
                     "unfused chain launch");
}
int lsfa_unfused_chain_num_launches(void) { return lsfa::unfused_chain_launches(); }

int lsfa_choose_feat_f32(const float* conv_feat, const float* conv_feat_prop, const uint8_t* eq_flag, float* out,
                         int N, long long per_frame, void* stream) {
  if (!conv_feat || !conv_feat_prop || !eq_flag || !out) return fail(LSFA_E_BADARG, "NULL pointer");
  if (N <= 0 || per_frame <= 0) return fail(LSFA_E_SHAPE, "non-positive dims");
  return cuda_result(lsfa::launch_choose_feat(conv_feat, conv_feat_prop, eq_flag, out, per_frame,
                                              (long long)N * per_frame, as_stream(stream)),
                     "choose_feat launch");
}

int lsfa_blend_logits_f32(const float* src0, const float* cur, const float* logits, const uint8_t* bypass, float* out,
                          int N, int C, int H, int W, void* stream) {
  if (!src0 || !cur || !logits || !out) return fail(LSFA_E_BADARG, "NULL pointer");
  if (N <= 0 || C <= 0 || H <= 0 || W <= 0) return fail(LSFA_E_SHAPE, "non-positive dims");
  return cuda_result(lsfa::launch_blend_logits(src0, cur, logits, bypass, out, N, C, H * W, as_stream(stream)),
                     "blend_logits launch");
}

size_t lsfa_mv_accumulate_workspace_bytes(int N, int height, int width) {
  if (N <= 0 || height <= 0 || width <= 0) return 0;
  return (size_t)N * height * width * (2 * 8 + 4);      // two (x,y) int2 fields + the owner map
}

size_t lsfa_mv_accumulate_trace_workspace_bytes(int N, int T, int height, int width) {
  if (N <= 0 || T < 0 || height <= 0 || width <= 0) return 0;
  return lsfa::mvacc_trace_workspace_bytes(N, T, height, width);
}

int lsfa_mv_accumulate_algo_i32(const int32_t* mvs, const int32_t* counts, int N, int T, int M, int height, int width,
                                int32_t* mv_out, void* workspace, size_t workspace_bytes, int algo, void* stream) {
  if (!mvs || !counts || !mv_out || !workspace) return fail(LSFA_E_BADARG, "NULL pointer");
  if (algo < 0 || algo > 2) return fail(LSFA_E_BADARG, "algo must be 0 (auto), 1 (per-frame field) or 2 (cell-index back-trace)");
  if (N <= 0 || T < 0 || M <= 0 || height <= 0 || width <= 0 || N > 65535 || height > 65535 ||
      (long long)height * width >= (1LL << 31))
    return fail(LSFA_E_SHAPE, "bad dims (N and height index the launch grid: at most 65535; height*width < 2^31)");
  const size_t need_field = lsfa_mv_accumulate_workspace_bytes(N, height, width);
  const size_t need_trace = (long long)N * T <= 65535 ? lsfa::mvacc_trace_workspace_bytes(N, T, height, width) : (size_t)-1;
  const size_t need = algo == 1 ? need_field : (algo == 2 ? need_trace : (need_trace < need_field ? need_trace : need_field));
  if (need == (size_t)-1) return fail(LSFA_E_UNSUPPORTED, "the back-trace form indexes its launch grid by N*T: at most 65535");
  if (workspace_bytes < need) return fail(LSFA_E_BADARG, "workspace too small: need %zu bytes", need);
  if ((reinterpret_cast<uintptr_t>(workspace) % 8) || (reinterpret_cast<uintptr_t>(mv_out) % 8) ||
      (reinterpret_cast<uintptr_t>(mvs) % 8))
    return fail(LSFA_E_ALIGN, "mvs, workspace and mv_out must be 8-byte aligned");
  cudaError_t e = lsfa::launch_mv_accumulate(mvs, counts, N, T, M, height, width, mv_out, workspace, workspace_bytes, algo, as_stream(stream));
  if (e == cudaErrorNotSupported) {
    cudaGetLastError();
    return fail(LSFA_E_UNSUPPORTED, "the requested algorithm cannot serve these arguments (workspace size or N*T)");
  }
  return cuda_result(e, "mv_accumulate launch");
}

int lsfa_mv_accumulate_i32(const int32_t* mvs, const int32_t* counts, int N, int T, int M, int height, int width,
                           int32_t* mv_out, void* workspace, size_t workspace_bytes, void* stream) {
  return lsfa_mv_accumulate_algo_i32(mvs, counts, N, T, M, height, width, mv_out, workspace, workspace_bytes, 0, stream);
}

int lsfa_coviar_residual_u8(const uint8_t* iframe, const uint8_t* cur, const int32_t* mv, int32_t* res, int N, int height,
                            int width, void* stream) {
  if (!iframe || !cur || !mv || !res) return fail(LSFA_E_BADARG, "NULL pointer");
  if (N <= 0 || height <= 0 || width <= 0 || N > 65535 || height > 65535)
    return fail(LSFA_E_SHAPE, "bad dims (N and height index the launch grid: at most 65535)");
  if (reinterpret_cast<uintptr_t>(mv) % 8) return fail(LSFA_E_ALIGN, "mv must be 8-byte aligned");
  return cuda_result(lsfa::launch_coviar_residual(iframe, cur, mv, res, N, height, width, as_stream(stream)),
                     "coviar_residual launch");
}

static int sampler_backward_common(const float* data, const float* coords, int is_flow, const float* og, float* gdata,
                                   float* ggrid, int N, int C, int Hi, int Wi, int Ho, int Wo, int req_data,
                                   int req_grid, void* workspace, size_t workspace_bytes, int kernel, void* stream) {
  if (!valid_req(req_data) || !valid_req(req_grid)) return fail(LSFA_E_BADARG, "unknown req %d / %d", req_data, req_grid);
  if (kernel < 0 || kernel > 2) return fail(LSFA_E_BADARG, "kernel must be 0 (auto), 1 (scatter) or 2 (gather)");
  if (N <= 0 || C <= 0 || Hi <= 0 || Wi <= 0 || Ho <= 0 || Wo <= 0)
    return fail(LSFA_E_SHAPE, "non-positive dims N=%d C=%d in %dx%d out %dx%d", N, C, Hi, Wi, Ho, Wo);
  if ((long long)Hi * Wi >= (1LL << 24) || (long long)Ho * Wo >= (1LL << 24))
    return fail(LSFA_E_SHAPE, "planes of 2^24 pixels or more are not supported");
  if (req_data == LSFA_REQ_NULL) gdata = nullptr;
  if (req_grid == LSFA_REQ_NULL) ggrid = nullptr;
  if (!gdata && !ggrid) return LSFA_OK;                        // nothing requested
  if (!data || !coords || !og) return fail(LSFA_E_BADARG, "data, grid/flow and out_grad are required");
  cudaError_t e = lsfa::launch_sampler_backward(data, coords, is_flow, og, gdata, ggrid, N, C, Hi, Wi, Ho, Wo,
                                                req_data == LSFA_REQ_ADD, req_grid == LSFA_REQ_ADD, half_extent(Wo),
                                                half_extent(Ho), workspace, workspace_bytes, kernel, as_stream(stream));
  if (e == cudaErrorNotSupported) {
    cudaGetLastError();
    return fail(LSFA_E_UNSUPPORTED, "the gather kernel cannot serve these arguments (workspace, plane size or alignment)");
  }
  return cuda_result(e, "sampler backward launch");
}

size_t lsfa_bilinear_sampler_backward_workspace_bytes(int N, int C, int Hi, int Wi, int Ho, int Wo) {
  (void)C;
  if (N <= 0 || Hi <= 0 || Wi <= 0 || Ho <= 0 || Wo <= 0) return 0;
  return lsfa::bwd_workspace_bytes(N, Hi * Wi, Ho * Wo);
}

int lsfa_bilinear_sampler_backward_f32(const float* data, const float* grid, const float* out_grad, float* grad_data,
                                       float* grad_grid, int N, int C, int Hi, int Wi, int Ho, int Wo, int req_data,
                                       int req_grid, void* workspace, size_t workspace_bytes, int kernel, void* stream) {
  return sampler_backward_common(data, grid, 0, out_grad, grad_data, grad_grid, N, C, Hi, Wi, Ho, Wo, req_data, req_grid,
                                 workspace, workspace_bytes, kernel, stream);
}

int lsfa_bilinear_sampler_backward_num_launches(int N, int C, int Hi, int Wi, int Ho, int Wo, int req_data, int req_grid,
                                                size_t workspace_bytes, int kernel) {
  if (N <= 0 || C <= 0 || Hi <= 0 || Wi <= 0 || Ho <= 0 || Wo <= 0) return 0;
  if (req_data == LSFA_REQ_NULL && req_grid == LSFA_REQ_NULL) return 0;
  return lsfa::sampler_backward_num_launches(N, C, Hi, Wi, Ho, Wo, req_data != LSFA_REQ_NULL,
                                             workspace_bytes >= lsfa::bwd_workspace_bytes(N, Hi * Wi, Ho * Wo), kernel);
}

int lsfa_grid_generator_warp_backward_f32(const float* grad_grid, float* grad_flow, int N, int H, int W, int req,
                                          void* stream) {
  if (!valid_req(req)) return fail(LSFA_E_BADARG, "unknown req %d", req);
  if (N <= 0 || H <= 0 || W <= 0) return fail(LSFA_E_SHAPE, "non-positive dims N=%d H=%d W=%d", N, H, W);
  if (req == LSFA_REQ_NULL) return LSFA_OK;
  if (!grad_grid || !grad_flow) return fail(LSFA_E_BADARG, "grad_grid and grad_flow are required");
  return cuda_result(lsfa::launch_grid_generator_backward(grad_grid, grad_flow, N, H, W, half_extent(W), half_extent(H),
                                                          req == LSFA_REQ_ADD, as_stream(stream)),
                     "grid_generator backward launch");
}

int lsfa_warp_backward_f32(const float* key, const float* flow, const float* out_grad, float* grad_key, float* grad_flow,
                           int N, int C, int H, int W, int req_key, int req_flow, void* workspace, size_t workspace_bytes,
                           int kernel, void* stream) {
  return sampler_backward_common(key, flow, 1, out_grad, grad_key, grad_flow, N, C, H, W, H, W, req_key, req_flow,
                                 workspace, workspace_bytes, kernel, stream);
}

int lsfa_nchw_to_nhwc(const float* src, void* dst, int N, int C, int H, int W, int dst_layout, void* stream) {
  if (!src || !dst) return fail(LSFA_E_BADARG, "NULL pointer");
  if (N <= 0 || C <= 0 || H <= 0 || W <= 0 || N > 65535) return fail(LSFA_E_SHAPE, "bad dims");
  if (dst_layout != LSFA_LAYOUT_NHWC_F32 && dst_layout != LSFA_LAYOUT_NHWC_BF16) return fail(LSFA_E_BADARG, "dst_layout must be NHWC");
  return cuda_result(lsfa::launch_nchw_to_nhwc(src, dst, N, C, H * W, dst_layout == LSFA_LAYOUT_NHWC_BF16,
                                               as_stream(stream)),
                     "nchw_to_nhwc launch");
}
int lsfa_nhwc_to_nchw(const void* src, float* dst, int N, int C, int H, int W, int src_layout, void* stream) {
  if (!src || !dst) return fail(LSFA_E_BADARG, "NULL pointer");
  if (N <= 0 || C <= 0 || H <= 0 || W <= 0 || N > 65535) return fail(LSFA_E_SHAPE, "bad dims");
  if (src_layout != LSFA_LAYOUT_NHWC_F32 && src_layout != LSFA_LAYOUT_NHWC_BF16) return fail(LSFA_E_BADARG, "src_layout must be NHWC");
  return cuda_result(lsfa::launch_nhwc_to_nchw(src, dst, N, C, H * W, src_layout == LSFA_LAYOUT_NHWC_BF16,
                                               as_stream(stream)),
                     "nhwc_to_nchw launch");
}

// ---------------------------------------------------------------------------------------------------------
// record / replay: the entry points only enqueue, so a frame's sequence of calls is one CUDA graph
// ---------------------------------------------------------------------------------------------------------
struct LsfaGraph {
  cudaGraph_t graph;
  cudaGraphExec_t exec;
};
int lsfa_graph_begin(void* stream) {
  if (!stream) return fail(LSFA_E_BADARG, "capture needs an explicit (non-NULL) stream");
  return cuda_result(cudaStreamBeginCapture(as_stream(stream), cudaStreamCaptureModeThreadLocal), "cudaStreamBeginCapture");
}
int lsfa_graph_end(void* stream, void** graph) {
  if (!graph) return fail(LSFA_E_BADARG, "graph out-pointer is NULL");
  *graph = nullptr;
  if (!stream) return fail(LSFA_E_BADARG, "capture needs an explicit (non-NULL) stream");
  cudaGraph_t g = nullptr;
  if (int r = cuda_result(cudaStreamEndCapture(as_stream(stream), &g), "cudaStreamEndCapture")) return r;
  if (!g) return fail(LSFA_E_CUDA, "the capture was invalidated by an error between lsfa_graph_begin and lsfa_graph_end");
  cudaGraphExec_t ex = nullptr;
  cudaError_t e = cudaGraphInstantiate(&ex, g, 0);
  if (e != cudaSuccess) {
    cudaGraphDestroy(g);
    return cuda_result(e, "cudaGraphInstantiate");
  }
  LsfaGraph* h = new (std::nothrow) LsfaGraph{g, ex};
  if (!h) {
    cudaGraphExecDestroy(ex);
    cudaGraphDestroy(g);
    return fail(LSFA_E_BADARG, "out of host memory");
  }
  *graph = h;
  return LSFA_OK;
}
int lsfa_graph_launch(void* graph, void* stream) {
  if (!graph) return fail(LSFA_E_BADARG, "graph is NULL");
  return cuda_result(cudaGraphLaunch(static_cast<LsfaGraph*>(graph)->exec, as_stream(stream)), "cudaGraphLaunch");
}
int lsfa_graph_destroy(void* graph) {
  if (!graph) return LSFA_OK;
  LsfaGraph* h = static_cast<LsfaGraph*>(graph);
  cudaGraphExecDestroy(h->exec);
  cudaGraphDestroy(h->graph);
  delete h;
  return LSFA_OK;
}

// ---------------------------------------------------------------------------------------------------------
// SURVEY 8f rank 2: the embedding / quality networks on tensor cores (conv_gemm_tc.cu)
// ---------------------------------------------------------------------------------------------------------
static int tc_sm_count() {
  int dev = 0, n = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0)
    return 148;
  return n;
}
static int tc_result(const char* msg, const char* what) {
  if (msg) return fail(LSFA_E_UNSUPPORTED, "%s: %s", what, msg);
  return cuda_result(cudaPeekAtLastError(), what);
}

int lsfa_pack_conv_weight_bf16(const float* w, void* w_packed, int Cout, int Cin, int ksize, void* stream) {
  if (!w || !w_packed) return fail(LSFA_E_BADARG, "NULL pointer");
  if (Cout <= 0 || Cin <= 0 || (ksize != 1 && ksize != 3)) return fail(LSFA_E_SHAPE, "bad dims (ksize must be 1 or 3)");
  lsfa::tc::launch_pack_weight(w, w_packed, Cout, Cin, ksize * ksize, as_stream(stream));
  return cuda_result(cudaPeekAtLastError(), "pack_conv_weight launch");
}

int lsfa_conv_bf16_nhwc(const void* x, const void* w_packed, const float* bias, void* out, int NB, int H, int W, int Cin,
                        int Cout, int ksize, int relu, void* stream) {
  if (!x || !w_packed || !bias || !out) return fail(LSFA_E_BADARG, "NULL pointer");
  if (NB <= 0 || H <= 0 || W <= 0 || Cin <= 0 || Cout <= 0) return fail(LSFA_E_SHAPE, "non-positive dims");
  if (ksize != 1 && ksize != 3) return fail(LSFA_E_SHAPE, "ksize must be 1 or 3");
  if (reinterpret_cast<uintptr_t>(out) & 15) return fail(LSFA_E_ALIGN, "out must be 16-byte aligned");
  lsfa::tc::ConvParams P{};
  P.NB = NB; P.H = H; P.W = W; P.Cin = Cin; P.Cout = Cout; P.taps = ksize * ksize;
  P.bias = bias;
  P.out = static_cast<__nv_bfloat16*>(out);
  return tc_result(lsfa::tc::launch_conv(x, w_packed, P, relu ? lsfa::tc::EPI_STORE_RELU : lsfa::tc::EPI_STORE, tc_sm_count(),
                                         as_stream(stream)),
                   "conv_bf16_nhwc");
}

static size_t align256(size_t v) { return (v + 255) & ~(size_t)255; }

size_t lsfa_embed_cosine_logits_workspace_bytes(int N, int H, int W, int C1, int C2, int E) {
  if (N <= 0 || H <= 0 || W <= 0 || C1 <= 0 || C2 <= 0 || E <= 0) return 0;
  const size_t px = (size_t)2 * N * H * W;
  return align256(px * C1 * 2) + align256(px * C2 * 2) + align256((size_t)(E / 256) * 2 * 3 * N * H * W * 4);
}

int lsfa_embed_cosine_logits_bf16_nhwc(const void* x, const void* w1, const float* b1, const void* w2, const float* b2,
                                       const void* w3, const float* b3, float* logits, int N, int H, int W, int C, int C1,
                                       int C2, int E, void* workspace, size_t workspace_bytes, void* stream) {
  if (!x || !w1 || !b1 || !w2 || !b2 || !w3 || !b3 || !logits || !workspace) return fail(LSFA_E_BADARG, "NULL pointer");
  if (N <= 0 || H <= 0 || W <= 0 || C <= 0 || C1 <= 0 || C2 <= 0 || E <= 0) return fail(LSFA_E_SHAPE, "non-positive dims");
  if (E % 256) return fail(LSFA_E_SHAPE, "E must be a multiple of 256");
  const size_t need = lsfa_embed_cosine_logits_workspace_bytes(N, H, W, C1, C2, E);
  if (workspace_bytes < need) return fail(LSFA_E_BADARG, "workspace too small: need %zu bytes", need);
  if (reinterpret_cast<uintptr_t>(workspace) & 255) return fail(LSFA_E_ALIGN, "workspace must be 256-byte aligned");
  const size_t px = (size_t)2 * N * H * W;
  char* ws = static_cast<char*>(workspace);
  __nv_bfloat16* h1 = reinterpret_cast<__nv_bfloat16*>(ws);
  __nv_bfloat16* h2 = reinterpret_cast<__nv_bfloat16*>(ws + align256(px * C1 * 2));
  float* partial = reinterpret_cast<float*>(ws + align256(px * C1 * 2) + align256(px * C2 * 2));
  const int sms = tc_sm_count();
  cudaStream_t st = as_stream(stream);
  lsfa::tc::ConvParams P{};
  P.NB = 2 * N; P.H = H; P.W = W;
  // em_conv1 + em_ReLU1 (SYM:119-121)
  P.Cin = C; P.Cout = C1; P.taps = 1; P.bias = b1; P.out = h1;
  if (int r = tc_result(lsfa::tc::launch_conv(x, w1, P, lsfa::tc::EPI_STORE_RELU, sms, st), "em_conv1")) return r;
  // em_conv2 + em_ReLU2 (SYM:123-125)
  P.Cin = C1; P.Cout = C2; P.taps = 9; P.bias = b2; P.out = h2;
  if (int r = tc_result(lsfa::tc::launch_conv(h1, w2, P, lsfa::tc::EPI_STORE_RELU, sms, st), "em_conv2")) return r;
  // em_conv3 (SYM:127-128) with compute_weight's reductions (SYM:111-116) as its epilogue
  P.Cin = C2; P.Cout = E; P.taps = 1; P.bias = b3; P.out = nullptr; P.partial = partial;
  if (int r = tc_result(lsfa::tc::launch_conv(h2, w3, P, lsfa::tc::EPI_COSINE, sms, st), "em_conv3+cosine")) return r;
  lsfa::tc::launch_cosine_finalize(partial, logits, 2 * (E / 256), N, H * W, st);   // two column halves per 256-channel chunk
  return cuda_result(cudaPeekAtLastError(), "cosine finalize launch");
}

int lsfa_nq_logits_bf16_nhwc(const void* x, const void* w1, const float* b1, const float* w2, const float* b2, const float* w3,
                             const float* b3, float* logits, int N, int H, int W, int C, void* stream) {
  if (!x || !w1 || !b1 || !w2 || !b2 || !w3 || !b3 || !logits) return fail(LSFA_E_BADARG, "NULL pointer");
  if (N <= 0 || H <= 0 || W <= 0 || C <= 0) return fail(LSFA_E_SHAPE, "non-positive dims");
  lsfa::tc::ConvParams P{};
  P.NB = 2 * N; P.H = H; P.W = W; P.Cin = C; P.Cout = 256; P.taps = 9;
  P.bias = b1; P.logits = logits; P.nq_w2 = w2; P.nq_b2 = b2; P.nq_w3 = w3; P.nq_b3 = b3;
  return tc_result(lsfa::tc::launch_conv(x, w1, P, lsfa::tc::EPI_NQ, tc_sm_count(), as_stream(stream)), "nq_logits");
}

// ---------------------------------------------------------------------------------------------------------
// backward of the fused operator's tails (aggregate_backward.cu) + a7/a8 backward (sampler_backward.cu)
// ---------------------------------------------------------------------------------------------------------
namespace {
struct BwdPlan {
  bool want_key, want_flow, want_scale, want_cur, want_logits, want_res, want_rnet, want_gw, pool_flow, want_emb;
  size_t tail_ws, flow_ws, samp_ws, cos_ws;
};
inline bool wanted(const void* p, int req) { return p != nullptr && req != LSFA_REQ_NULL; }
// the LsfaAggGrads of binaries built before the embedding gradients existed
constexpr size_t kAggGradsV1Bytes = offsetof(LsfaAggGrads, grad_emb_warp);
// COSINE mode: [logits (N,2,H,W)][d/d(logits) (N,2,H,W)][cosine backward scratch], after the other regions
size_t cosine_bwd_plane_bytes(const LsfaAggArgs* a) { return ((size_t)a->N * 2 * a->H * a->W * 4 + 255) & ~(size_t)255; }
// Validate fwd and grads; G = *g with the fields an older struct lacks read as NULL / 0.
int plan_backward(const LsfaAggArgs* a, const LsfaAggGrads* g, BwdPlan& B, LsfaAggGrads& G) {
  if (!a || !g) return fail(LSFA_E_BADARG, "fwd and grads are required");
  if (g->struct_bytes != (int32_t)sizeof(LsfaAggGrads) && g->struct_bytes != (int32_t)kAggGradsV1Bytes)
    return fail(LSFA_E_BADARG, "grads->struct_bytes=%d, expected %zu (or %zu without the embedding gradients)", g->struct_bytes,
                sizeof(LsfaAggGrads), kAggGradsV1Bytes);
  memset(&G, 0, sizeof(G));
  memcpy(&G, g, (size_t)g->struct_bytes);
  g = &G;
  if (a->struct_bytes != (int32_t)sizeof(LsfaAggArgs)) return fail(LSFA_E_BADARG, "fwd->struct_bytes=%d, expected %zu", a->struct_bytes, sizeof(LsfaAggArgs));
  if (a->layout != LSFA_LAYOUT_NCHW_F32) return fail(LSFA_E_UNSUPPORTED, "the backward is built for the NCHW float32 layout");
  const int reqs[8] = {g->req_key, g->req_flow, g->req_scale, g->req_cur, g->req_logits, g->req_res, g->req_rnet, g->req_emb};
  for (int r : reqs) if (!valid_req(r)) return fail(LSFA_E_BADARG, "unknown req %d", r);
  const bool cosine = a->weight_mode == LSFA_W_COSINE;
  B.want_emb = wanted(g->grad_emb_warp, g->req_emb) || wanted(g->grad_emb_cur, g->req_emb);
  if (B.want_emb && !cosine) return fail(LSFA_E_BADARG, "embedding gradients requested but weight_mode is not COSINE");
  if (cosine && wanted(g->grad_logits, g->req_logits))
    return fail(LSFA_E_BADARG, "grad_logits requested in COSINE mode: the logits are computed from the embeddings, not an input");
  if (cosine && (!a->emb_warp || !a->emb_cur || a->E <= 0)) return fail(LSFA_E_BADARG, "COSINE mode needs emb_warp, emb_cur and E > 0");
  B.want_key = wanted(g->grad_key, g->req_key);
  B.want_flow = wanted(g->grad_flow, g->req_flow);
  B.want_scale = wanted(g->grad_scale, g->req_scale);
  B.want_cur = wanted(g->grad_cur, g->req_cur);
  B.want_logits = wanted(g->grad_logits, g->req_logits) || B.want_emb;   // COSINE: d/d(logits) into the workspace
  B.want_res = wanted(g->grad_res, g->req_res);
  B.want_rnet = wanted(g->grad_rnet_w, g->req_rnet);
  if (B.want_rnet && !g->grad_rnet_b) return fail(LSFA_E_BADARG, "grad_rnet_w and grad_rnet_b go together");
  if (B.want_scale && !a->scale_map) return fail(LSFA_E_BADARG, "grad_scale requested but the forward had no scale_map");
  if (B.want_cur && a->weight_mode == LSFA_W_NONE) return fail(LSFA_E_BADARG, "grad_cur requested but weight_mode is NONE");
  if (B.want_logits && a->weight_mode != LSFA_W_LOGITS && !cosine) return fail(LSFA_E_BADARG, "grad_logits requested but weight_mode is not LOGITS");
  if ((B.want_res || B.want_rnet) && !a->res) return fail(LSFA_E_BADARG, "residual gradients requested but the forward had no res");
  if (B.want_flow && a->flow_kind != LSFA_FLOW_PREPOOLED && a->flow_kind != LSFA_FLOW_GRID)
    return fail(LSFA_E_BADARG, "grad_flow needs LSFA_FLOW_PREPOOLED or LSFA_FLOW_GRID: raw motion vectors are integer data (SYM:319-321)");
  if (B.want_key || B.want_flow) {
    if (a->key_index) return fail(LSFA_E_UNSUPPORTED, "grad_key / grad_flow need private keys (key_index NULL)");
    if (a->flow_kind == LSFA_FLOW_COVIAR_I32) return fail(LSFA_E_UNSUPPORTED, "grad_key with LSFA_FLOW_COVIAR_I32: prepare and pool the MV first");
    const int Hk = a->key_h > 0 ? a->key_h : a->H, Wk = a->key_w > 0 ? a->key_w : a->W;
    if (a->flow_kind != LSFA_FLOW_GRID && (Hk != a->H || Wk != a->W)) return fail(LSFA_E_UNSUPPORTED, "grad_key with a flow needs key planes of the output's size");
  }
  if (a->N <= 0 || a->C <= 0 || a->H <= 0 || a->W <= 0) return fail(LSFA_E_SHAPE, "non-positive dims");
  B.want_gw = B.want_key || B.want_flow;
  B.pool_flow = B.want_gw && (a->flow_kind == LSFA_FLOW_RAW_I32 || a->flow_kind == LSFA_FLOW_RAW_F32);
  const int HW = a->H * a->W;
  B.tail_ws = lsfa::tail_backward_workspace_bytes(a->N, a->C, HW, B.want_gw, B.want_logits, B.want_res || B.want_rnet);
  B.flow_ws = B.pool_flow ? (((size_t)a->N * 2 * HW * 4 + 255) & ~(size_t)255) : 0;
  const int Hk = a->key_h > 0 ? a->key_h : a->H, Wk = a->key_w > 0 ? a->key_w : a->W;
  B.samp_ws = B.want_gw ? ((lsfa::bwd_workspace_bytes(a->N, Hk * Wk, HW) + 255) & ~(size_t)255) : 0;
  B.cos_ws = cosine ? 2 * cosine_bwd_plane_bytes(a) + lsfa::cosine_backward_workspace_bytes(a->N, a->E, HW) : 0;
  return LSFA_OK;
}

}  // namespace

size_t lsfa_warp_scale_aggregate_backward_workspace_bytes(const LsfaAggArgs* fwd, const LsfaAggGrads* grads) {
  BwdPlan B;
  LsfaAggGrads G;
  if (plan_backward(fwd, grads, B, G) != LSFA_OK) return 0;
  return B.tail_ws + B.flow_ws + B.samp_ws + B.cos_ws;
}

int lsfa_warp_scale_aggregate_backward_f32_nchw(const LsfaAggArgs* fwd, const LsfaAggGrads* grads, void* stream) {
  BwdPlan B;
  LsfaAggGrads G;
  if (int r = plan_backward(fwd, grads, B, G)) return r;
  const LsfaAggGrads* g = &G;
  if (!g->out_grad) return fail(LSFA_E_BADARG, "out_grad is required");
  lsfa::AggParams P;
  if (int r = build_params(fwd, P)) return r;
  if (P.HWk > 16383) return fail(LSFA_E_UNSUPPORTED, "key planes above 16,383 pixels are not supported by the backward");
  const size_t need = B.tail_ws + B.flow_ws + B.samp_ws + B.cos_ws;
  if (!g->workspace || g->workspace_bytes < need) return fail(LSFA_E_BADARG, "workspace too small: need %zu bytes", need);
  if (reinterpret_cast<uintptr_t>(g->workspace) & 255) return fail(LSFA_E_ALIGN, "workspace must be 256-byte aligned");
  cudaStream_t st = as_stream(stream);
  char* ws = static_cast<char*>(g->workspace);
  float* glogits = g->grad_logits;
  char* cos_ws = ws + B.tail_ws + B.flow_ws + B.samp_ws;
  const size_t plane_b = fwd->weight_mode == LSFA_W_COSINE ? cosine_bwd_plane_bytes(fwd) : 0;
  const bool tma_sums = fwd->force_generic != 1;
  if (fwd->weight_mode == LSFA_W_COSINE) {
    // the forward's logits, then the LOGITS-mode backward on them with d/d(logits) kept in the workspace
    float* lg = reinterpret_cast<float*>(cos_ws);
    glogits = reinterpret_cast<float*>(cos_ws + plane_b);
    if (int r = cuda_result(cosine_logits_nchw(static_cast<const float*>(fwd->emb_warp), static_cast<const float*>(fwd->emb_cur), lg,
                                               fwd->N, fwd->E, P.HW, cos_ws + 2 * plane_b, B.cos_ws - 2 * plane_b, tma_sums, st),
                            "cosine_logits_nchw launch"))
      return r;
    P.mode = LSFA_W_LOGITS;
    P.logits = lg;
  }
  float* gw = nullptr;
  lsfa::TailBwdRequest R{};
  R.out_grad = g->out_grad;
  R.grad_scale = B.want_scale ? g->grad_scale : nullptr; R.add_scale = g->req_scale == LSFA_REQ_ADD;
  R.grad_cur = B.want_cur ? g->grad_cur : nullptr;       R.add_cur = g->req_cur == LSFA_REQ_ADD;
  R.grad_logits = B.want_logits ? glogits : nullptr;     R.add_logits = B.want_emb ? 0 : g->req_logits == LSFA_REQ_ADD;
  R.grad_res = B.want_res ? g->grad_res : nullptr;       R.add_res = g->req_res == LSFA_REQ_ADD;
  R.grad_rnet_w = B.want_rnet ? g->grad_rnet_w : nullptr; R.grad_rnet_b = B.want_rnet ? g->grad_rnet_b : nullptr;
  R.add_rnet = g->req_rnet == LSFA_REQ_ADD;
  R.want_gw = B.want_gw;
  R.gw_out = &gw;
  if (int r = cuda_result(lsfa::launch_tail_backward(P, R, ws, st), "tail backward launch")) return r;
  if (B.want_emb) {
    const bool add = g->req_emb == LSFA_REQ_ADD;
    if (int r = cuda_result(lsfa::launch_cosine_backward_nchw(static_cast<const float*>(fwd->emb_warp), static_cast<const float*>(fwd->emb_cur),
                                                              glogits, fwd->bypass, g->grad_emb_warp, g->grad_emb_cur, add, add, fwd->N,
                                                              fwd->E, P.HW, cos_ws + 2 * plane_b, B.cos_ws - 2 * plane_b, tma_sums, 0, st),
                            "cosine backward launch"))
      return r;
  }
  if (!B.want_gw) return LSFA_OK;
  ws += B.tail_ws;
  const float* coords = static_cast<const float*>(fwd->flow);
  int is_flow = fwd->flow_kind != LSFA_FLOW_GRID;
  if (B.pool_flow) {                         // a3+a5+a6 once more: the sampler's backward wants the pooled flow
    float* pooled = reinterpret_cast<float*>(ws);
    ws += B.flow_ws;
    if (int r = cuda_result(lsfa::launch_mv_pool(fwd->flow, fwd->flow_kind == LSFA_FLOW_RAW_I32, pooled, fwd->N, fwd->mv_h, fwd->mv_w, fwd->H,
                                                 fwd->W, fwd->im_scale / 16.0, fwd->pool_mode, st), "mv_pool launch")) return r;
    coords = pooled;
  }
  const int Hk = fwd->key_h > 0 ? fwd->key_h : fwd->H, Wk = fwd->key_w > 0 ? fwd->key_w : fwd->W;
  return sampler_backward_common(static_cast<const float*>(fwd->key), coords, is_flow, gw, B.want_key ? g->grad_key : nullptr,
                                 B.want_flow ? g->grad_flow : nullptr, fwd->N, fwd->C, Hk, Wk, fwd->H, fwd->W,
                                 B.want_key ? g->req_key : LSFA_REQ_NULL, B.want_flow ? g->req_flow : LSFA_REQ_NULL, ws, B.samp_ws, 0, stream);
}

}  // extern "C"
