// Device-side building blocks shared by every kernel of the path (sm_100a only).
//
//  * exact_*   : the integer / indexing math of GridGenerator(warp) + BilinearSampler in
//                the reference's float32 op order, written with round-to-nearest intrinsics
//                so ptxas can neither contract to FMA nor re-associate (SURVEY.md section 7
//                "fp32 coordinate round trip").
//  * pool_*    : the stride-16 reduction of lib/utils/image.py:220-228 in float64.
//  * mbar_* / bulk_g2s : mbarrier + cp.async.bulk (TMA bulk copy, SASS UBLKCP) wrappers.
//  * ld/st helpers with cache hints for once-touched streams.
#pragma once
#include <cstdlib>

#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>

#include "../../include/lsfa_ops.h"

namespace lsfa {

// Ablation / experiment knobs (work-split percentages, kernel-shape overrides ...) are COMPILED OUT of the product build:
// the library's behaviour never depends on the environment.  Build with -DLSFA_EXPERIMENTS (LSFA_NVCC_EXTRA) to read them.
inline const char* knob(const char* name) {
#ifdef LSFA_EXPERIMENTS
  return getenv(name);
#else
  (void)name;
  return nullptr;
#endif
}

// ---------------------------------------------------------------------------------------
// Kernel-side view of LsfaAggArgs (plain values, passed by value as a __grid_constant__)
// ---------------------------------------------------------------------------------------
struct AggParams {
  int N, C, H, W, HW;          // output dims
  int Hk, Wk, HWk;             // key plane dims
  const void* key;
  const int* key_index;
  int num_keys;                // key features behind `key`: key_index values are clamped into [0, num_keys)
  int flow_kind;
  const void* flow;
  int mv_h, mv_w;
  double mv_scale;             // im_scale * (1/16)
  int src_h, src_w;            // LSFA_FLOW_COVIAR_I32: coviar image size (mv_h, mv_w = resized size)
  double inv_scale;            // 1 / im_scale
  int mv_negate, mv_hflip, mv_identity;
  int pool_mode;
  const void* scale;
  const float* res;
  const float* rnet_w;
  const float* rnet_b;
  const void* cur;
  int mode;
  const float* logits;
  const void* emb_warp;
  const void* emb_cur;
  int E;
  const unsigned char* bypass;
  void* out;
  int req_add;
  float half_w, half_h;        // (W-1)/2, (H-1)/2 of the flow grid (GridGenerator)
  float wk_m1, hk_m1;          // Wk-1, Hk-1 (BilinearSampler de-normalisation)
  // tiling of the plane-resident kernel
  int K;                       // channels per stage
  int chunks;                  // C / K
  int parts;                   // pixel parts per frame
  int part_pix;                // pixels per part (multiple of block size)
  int stages;
  unsigned stage_bytes;
  long long items;
  // stage layout of the all-TMA kernel: [key planes | scale chunk | cur/out chunk]
  unsigned key_bytes, io_bytes, off_scale, off_io;
  unsigned* sched;             // zeroed counter(s) for dynamic work claims, or NULL = static split
  long long pool_base;         // all-TMA kernel: items [0,pool_base) are split statically, the rest claimed from sched[0]
  const uint4* records;        // per-pixel packed sampling records (N*HW x 32 B) from the pre-pass, or NULL
  int canon;                   // the record pre-pass writes canonical_taps() records (warp-only variant of the all-TMA kernel)
  int records_ready;           // `records` already hold this launch's records (tail backward: the forward's folded weights)
  unsigned* zero_counter;      // record pre-pass: the streaming kernel's work-claim counter, zeroed here (saves a memset node)
  int coop;                    // all-TMA NCHW kernel launched cooperatively: its own consumers build the records, then a
                               // grid-wide barrier - the one-launch form for small batches (no pre-pass, no memset)
  int rnet_smem;               // channels-last tile kernel: rnet weights staged in dynamic shared memory
  int direct_store;            // all-TMA NCHW kernel, variants without cur: consumers store to global themselves
  unsigned* rowrange;          // 2 per (frame, pixel part), written by the pre-pass with atomicMax over zeros:
                               // [0] = last key row any tap of the part reads + 1, [1] = Hk - first such row; or NULL
};

// which key feature frame n samples (tile_as.py:16-19 without the tile).  A slot outside the table would make the
// bulk copies read whole planes from an arbitrary address, so it is clamped (memory safety; the host entry points that see
// the indices on the host - lsfa_host_aggregate_f32_nchw - reject them with an error instead)
__device__ __forceinline__ int key_slot(const AggParams& P, int n) {
  if (!P.key_index) return n;
  return min(max(__ldg(P.key_index + n), 0), P.num_keys - 1);
}

// ---------------------------------------------------------------------------------------
// a7: GridGenerator(warp)  -  grid = (flow + pos) / half - 1     (float32, add/div/sub)
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ float exact_grid(float flow, float pos, float half) {
  return __fsub_rn(__fdiv_rn(__fadd_rn(flow, pos), half), 1.0f);
}

// a8: real = (g + 1) * (dim - 1) / 2                              (float32, add/mul/div)
__device__ __forceinline__ float exact_denorm(float g, float dim_m1) {
  return __fdiv_rn(__fmul_rn(__fadd_rn(g, 1.0f), dim_m1), 2.0f);
}

// floor index with the same clamp the oracle applies to out-of-range / NaN coordinates
__device__ __forceinline__ int exact_floor_index(float real) {
  const float big = 16777216.0f;  // 2^24
  float f = floorf(real);
  if (!(f >= -big)) f = -big;     // also catches NaN
  if (f > big) f = big;
  return (int)f;
}

// top-left weight: w = float(1.0 - double(real - float(i0)))  (the literal 1.0 is a double)
__device__ __forceinline__ float exact_tl_weight(float real, int i0) {
  return (float)(1.0 - (double)__fsub_rn(real, (float)i0));
}

// One output pixel's sampling record.  Tap weights have invalid (out-of-plane) taps zeroed and
// are later pre-multiplied by the blend weight of the warped source (fold_blend); the four
// element indices are clamped into the plane so every tap address is always readable.
struct PixelRec {
  float w00, w01, w10, w11;   // bilinear weights (x ww after fold_blend)
  float ww, wc;               // blend weights of the warped source / the current feature
  int i00, i01, i10, i11;     // element offsets inside one key plane
  int edge;                   // bit 0: x0 < 0, bit 1: x0 > Wk-2, bit 2: y0 < 0, bit 3: y0 > Hk-2 (canonical_taps; window kernel: tap box origin)
};

__device__ __forceinline__ PixelRec make_taps(float gx, float gy, int Hk, int Wk, float wk_m1,
                                              float hk_m1) {
  const float xr = exact_denorm(gx, wk_m1);
  const float yr = exact_denorm(gy, hk_m1);
  const int x0 = exact_floor_index(xr);
  const int y0 = exact_floor_index(yr);
  const float wx = exact_tl_weight(xr, x0);
  const float wy = exact_tl_weight(yr, y0);
  const double owx = 1.0 - (double)wx, owy = 1.0 - (double)wy;
  const bool xl = (x0 >= 0) && (x0 <= Wk - 1);
  const bool xh = (x0 + 1 >= 0) && (x0 + 1 <= Wk - 1);
  const bool yl = (y0 >= 0) && (y0 <= Hk - 1);
  const bool yh = (y0 + 1 >= 0) && (y0 + 1 <= Hk - 1);
  PixelRec t;
  t.w00 = (xl && yl) ? (float)((double)wy * (double)wx) : 0.0f;
  t.w01 = (xh && yl) ? (float)((double)wy * owx) : 0.0f;
  t.w10 = (xl && yh) ? (float)(owy * (double)wx) : 0.0f;
  t.w11 = (xh && yh) ? (float)(owy * owx) : 0.0f;
  const int xa = min(max(x0, 0), Wk - 1), xb = min(max(x0 + 1, 0), Wk - 1);
  const int ya = min(max(y0, 0), Hk - 1), yb = min(max(y0 + 1, 0), Hk - 1);
  t.i00 = ya * Wk + xa;
  t.i01 = ya * Wk + xb;
  t.i10 = yb * Wk + xa;
  t.i11 = yb * Wk + xb;
  t.edge = (x0 < 0 ? 1 : 0) | (x0 > Wk - 2 ? 2 : 0) | (y0 < 0 ? 4 : 0) | (y0 > Hk - 2 ? 8 : 0);
  t.ww = 1.0f;
  t.wc = 0.0f;
  return t;
}

// Canonical form of a record for the shared-memory gather of the all-TMA NCHW kernels: the four taps become the 2x2
// block at ONE base offset (base, base+1, base+Wk, base+Wk+1), all inside the plane (needs Hk, Wk >= 2), so the inner
// loop needs one offset register per pixel and no unpacking.  At a plane border the block is shifted inwards and the
// weights move with their taps: the slot a tap leaves gets weight 0 (it already was 0: that tap lay outside the plane)
// and the non-zero terms keep their relative order in the fma chain of tap_chain(), so with finite key values the result
// is the same float (a zero-weight term adds exactly nothing).
__device__ __forceinline__ void canonical_taps(PixelRec& t, int Hk, int Wk) {
  const int y0 = t.i00 / Wk, x0 = t.i00 - y0 * Wk;        // clamped top-left tap
  const int bx = min(x0, Wk - 2), by = min(y0, Hk - 2);
  float a = t.w00, b = t.w01, c = t.w10, d = t.w11;
  if (t.edge & 1) { a = b; b = 0.0f; c = d; d = 0.0f; }   // left of the plane: the right column becomes the block's left one
  if (t.edge & 2) { b = a; a = 0.0f; d = c; c = 0.0f; }   // last column: the left column becomes the block's right one
  if (t.edge & 4) { a = c; b = d; c = 0.0f; d = 0.0f; }   // above the plane
  if (t.edge & 8) { c = a; d = b; a = 0.0f; b = 0.0f; }   // last row
  t.w00 = a; t.w01 = b; t.w10 = c; t.w11 = d;
  t.i00 = by * Wk + bx;
  t.i01 = t.i00 + 1;
  t.i10 = t.i00 + Wk;
  t.i11 = t.i10 + 1;
}

// Fold the warped source's blend weight into the tap weights: one multiply per pixel instead
// of one per element.  Exact for ww in {1, 0.5}; one extra rounding (<= 1 ulp) for softmax.
__device__ __forceinline__ void fold_blend(PixelRec& t, float ww, float wc) {
  t.ww = ww;
  t.wc = wc;
  t.w00 *= ww;
  t.w01 *= ww;
  t.w10 *= ww;
  t.w11 *= ww;
}

// The per-element arithmetic shared by every fp32 kernel (so they agree bit for bit):
//   v  = ww * bilinear(key)              (4-tap chain, weights pre-folded)
//   v  = v * scale                       [a9]
//   v += ww * (rw . res + rb)            [a10]
//   o  = wc * cur + v                    [a11-a14]
__device__ __forceinline__ float tap_chain(const PixelRec& t, float v00, float v01, float v10,
                                           float v11) {
  float v = t.w00 * v00;
  v = fmaf(t.w01, v01, v);
  v = fmaf(t.w10, v10, v);
  return fmaf(t.w11, v11, v);
}
__device__ __forceinline__ float rnet_term(float rw0, float rw1, float rw2, float rb, float r0,
                                           float r1, float r2) {
  float r = rw0 * r0;
  r = fmaf(rw1, r1, r);
  r = fmaf(rw2, r2, r);
  return r + rb;
}

// ---------------------------------------------------------------------------------------
// a3+a5+a6: stride-16 reduction of one (x|y) component of the raw MV image, float64.
// centre2x2: ((p[7,7]+p[7,8]) + (p[8,7]+p[8,8])) * 0.25, zero padding beyond (h,w).
// ---------------------------------------------------------------------------------------
template <typename T>
__device__ __forceinline__ double raw_at(const T* __restrict__ img, int h, int w, int nch,
                                         int y, int x, int ch) {
  if (y >= h || x >= w) return 0.0;
  return (double)__ldg(img + ((size_t)y * w + x) * nch + ch);
}

template <typename T>
__device__ __forceinline__ double pool_cell(const T* __restrict__ img, int h, int w, int nch,
                                            int cy, int cx, int ch, int mode) {
  const int y0 = cy * 16, x0 = cx * 16;
  if (mode == LSFA_POOL_CENTRE2X2) {
    const double a = raw_at(img, h, w, nch, y0 + 7, x0 + 7, ch);
    const double b = raw_at(img, h, w, nch, y0 + 7, x0 + 8, ch);
    const double c = raw_at(img, h, w, nch, y0 + 8, x0 + 7, ch);
    const double d = raw_at(img, h, w, nch, y0 + 8, x0 + 8, ch);
    return __dmul_rn(__dadd_rn(__dadd_rn(a, b), __dadd_rn(c, d)), 0.25);
  }
  double acc = 0.0;
#pragma unroll 1
  for (int r = 0; r < 16; ++r)
#pragma unroll 1
    for (int q = 0; q < 16; ++q) acc = __dadd_rn(acc, raw_at(img, h, w, nch, y0 + r, x0 + q, ch));
  return __dmul_rn(acc, 1.0 / 256.0);
}

// ---------------------------------------------------------------------------------------
// a1+a2 on the fly: one sample of the stage-1 image (sign, h-flip, cv2.resize INTER_LINEAR on
// float32: horizontal pass then vertical pass, no FMA) computed straight from coviar's int32
// array; zero beyond the resized image (the pad of image.py:207-215).
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ void linear_coeff(int d, int sn, double inv_scale, int& s, float& f) {
  f = (float)(__dsub_rn(__dmul_rn((double)d + 0.5, inv_scale), 0.5));
  const float fl = floorf(f);
  s = (int)fl;
  f = __fsub_rn(f, fl);
  if (s < 0) { s = 0; f = 0.f; }
  if (s >= sn - 1) { s = sn - 1; f = 0.f; }
}

__device__ __forceinline__ float coviar_src(const int* __restrict__ img, int w, int y, int x, int ch,
                                            int negate, int hflip) {
  const int xs = hflip ? (w - 1 - x) : x;
  float v = (float)__ldg(img + ((size_t)y * w + xs) * 2 + ch);
  if (negate) v = -v;
  if (hflip && ch == 0) v = -v;
  return v;
}

__device__ __forceinline__ float coviar_resized(const int* __restrict__ img, int h, int w, int oy, int ox,
                                                int ch, double inv_scale, int identity, int negate, int hflip) {
  if (identity) return coviar_src(img, w, oy, ox, ch, negate, hflip);
  int sx, sy;
  float fx, fy;
  linear_coeff(ox, w, inv_scale, sx, fx);
  linear_coeff(oy, h, inv_scale, sy, fy);
  const int sx1 = min(sx + 1, w - 1), sy1 = min(sy + 1, h - 1);
  const float a0 = __fsub_rn(1.0f, fx), b0 = __fsub_rn(1.0f, fy);
  const float t0 = __fadd_rn(__fmul_rn(coviar_src(img, w, sy, sx, ch, negate, hflip), a0),
                             __fmul_rn(coviar_src(img, w, sy, sx1, ch, negate, hflip), fx));
  const float t1 = __fadd_rn(__fmul_rn(coviar_src(img, w, sy1, sx, ch, negate, hflip), a0),
                             __fmul_rn(coviar_src(img, w, sy1, sx1, ch, negate, hflip), fx));
  return __fadd_rn(__fmul_rn(t0, b0), __fmul_rn(t1, fy));
}

// pooled (centre 2x2 | avg16) flow component of feature cell (y,x) straight from the coviar image
__device__ __forceinline__ double coviar_pool_cell(const AggParams& P, const int* __restrict__ img, int y, int x, int ch) {
  auto at = [&](int ry, int rx) -> double {
    if (ry >= P.mv_h || rx >= P.mv_w) return 0.0;
    return (double)coviar_resized(img, P.src_h, P.src_w, ry, rx, ch, P.inv_scale, P.mv_identity, P.mv_negate, P.mv_hflip);
  };
  if (P.pool_mode == LSFA_POOL_CENTRE2X2) {
    const double a = at(16 * y + 7, 16 * x + 7), b = at(16 * y + 7, 16 * x + 8);
    const double c = at(16 * y + 8, 16 * x + 7), d = at(16 * y + 8, 16 * x + 8);
    return __dmul_rn(__dadd_rn(__dadd_rn(a, b), __dadd_rn(c, d)), 0.25);
  }
  double acc = 0.0;
#pragma unroll 1
  for (int r = 0; r < 16; ++r)
#pragma unroll 1
    for (int q = 0; q < 16; ++q) acc = __dadd_rn(acc, at(16 * y + r, 16 * x + q));
  return __dmul_rn(acc, 1.0 / 256.0);
}

// flow (feature cells) of output pixel (y,x) of frame n from whatever the caller supplied;
// returns the normalised grid coordinates gx, gy.
__device__ __forceinline__ void pixel_grid(const AggParams& P, int n, int y, int x, float& gx,
                                           float& gy) {
  const int p = y * P.W + x;
  if (P.flow_kind == LSFA_FLOW_GRID) {
    const float* g = (const float*)P.flow + (size_t)n * 2 * P.HW;
    gx = __ldg(g + p);
    gy = __ldg(g + P.HW + p);
    return;
  }
  float fx, fy;
  if (P.flow_kind == LSFA_FLOW_PREPOOLED) {
    const float* f = (const float*)P.flow + (size_t)n * 2 * P.HW;
    fx = __ldg(f + p);
    fy = __ldg(f + P.HW + p);
  } else if (P.flow_kind == LSFA_FLOW_COVIAR_I32) {
    const int* mv = (const int*)P.flow + (size_t)n * P.src_h * P.src_w * 2;
    fx = (float)__dmul_rn(coviar_pool_cell(P, mv, y, x, 0), P.mv_scale);
    fy = (float)__dmul_rn(coviar_pool_cell(P, mv, y, x, 1), P.mv_scale);
  } else if (P.flow_kind == LSFA_FLOW_RAW_I32) {
    const int* mv = (const int*)P.flow + (size_t)n * P.mv_h * P.mv_w * 2;
    fx = (float)__dmul_rn(pool_cell(mv, P.mv_h, P.mv_w, 2, y, x, 0, P.pool_mode), P.mv_scale);
    fy = (float)__dmul_rn(pool_cell(mv, P.mv_h, P.mv_w, 2, y, x, 1, P.pool_mode), P.mv_scale);
  } else {
    const float* mv = (const float*)P.flow + (size_t)n * P.mv_h * P.mv_w * 2;
    fx = (float)__dmul_rn(pool_cell(mv, P.mv_h, P.mv_w, 2, y, x, 0, P.pool_mode), P.mv_scale);
    fy = (float)__dmul_rn(pool_cell(mv, P.mv_h, P.mv_w, 2, y, x, 1, P.pool_mode), P.mv_scale);
  }
  gx = exact_grid(fx, (float)x, P.half_w);
  gy = exact_grid(fy, (float)y, P.half_h);
}

// softmax over {l_warp, l_cur} as mx.sym.softmax: exp(x - max) / sum
__device__ __forceinline__ void softmax2(float lw, float lc, float& ww, float& wc) {
  const float m = fmaxf(lw, lc);
  const float ew = expf(lw - m), ec = expf(lc - m);
  const float s = ew + ec;
  ww = ew / s;
  wc = ec / s;
}

// per-pixel blend weights (ww on src0, wc on cur) for the non-cosine modes
__device__ __forceinline__ void pixel_weights(const AggParams& P, int n, int p, float& ww,
                                              float& wc) {
  ww = 1.0f;
  wc = 0.0f;
  if (P.mode == LSFA_W_ADD) {
    wc = 1.0f;
  } else if (P.mode == LSFA_W_MEAN) {
    ww = 0.5f;
    wc = 0.5f;
  } else if (P.mode == LSFA_W_LOGITS || P.mode == LSFA_W_COSINE) {
    const float* l = P.logits + (size_t)n * 2 * P.HW;
    softmax2(__ldg(l + p), __ldg(l + P.HW + p), ww, wc);
  }
}

// ---------------------------------------------------------------------------------------
// Split form of the record build: issue every global load of a pixel first (PixelLoads), do the
// arithmetic later (finish_pixel).  A thread that owns several pixels issues the loads of all of
// them back to back, so a record rebuild costs ONE trip to DRAM instead of two per pixel - under
// a saturated HBM that trip is 2-3 us and was the largest non-streaming cost of the fused kernel.
// ---------------------------------------------------------------------------------------
struct PixelLoads {
  unsigned t[8];   // raw MV: centre taps [row7: x7(ch0,ch1) x8(ch0,ch1)] [row8: ...]; flow/grid: t[0]=x, t[1]=y
  float l0, l1;    // logits (warp, cur)
};

__device__ __forceinline__ uint2 ldg_u2_or_zero(const void* base, size_t elem, bool ok) {
  uint2 v = make_uint2(0u, 0u);
  if (ok) v = __ldg(reinterpret_cast<const uint2*>(base) + elem);
  return v;
}

__device__ __forceinline__ PixelLoads issue_pixel_loads(const AggParams& P, int n, int y, int x) {
  PixelLoads L;
#pragma unroll
  for (int i = 0; i < 8; ++i) L.t[i] = 0u;
  L.l0 = L.l1 = 0.0f;
  const int p = y * P.W + x;
  if (P.flow_kind == LSFA_FLOW_GRID || P.flow_kind == LSFA_FLOW_PREPOOLED) {
    const float* f = (const float*)P.flow + (size_t)n * 2 * P.HW;
    L.t[0] = __float_as_uint(__ldg(f + p));
    L.t[1] = __float_as_uint(__ldg(f + P.HW + p));
  } else if (P.pool_mode == LSFA_POOL_CENTRE2X2 && P.flow_kind != LSFA_FLOW_COVIAR_I32) {
    // (x,y) pairs are 8 bytes: one 8-byte load per tap, zero beyond the unpadded image
    const char* img = (const char*)P.flow + (size_t)n * P.mv_h * P.mv_w * 8;
    const int y7 = 16 * y + 7, x7 = 16 * x + 7;
    const uint2 a = ldg_u2_or_zero(img, (size_t)y7 * P.mv_w + x7, y7 < P.mv_h && x7 < P.mv_w);
    const uint2 b = ldg_u2_or_zero(img, (size_t)y7 * P.mv_w + x7 + 1, y7 < P.mv_h && x7 + 1 < P.mv_w);
    const uint2 c = ldg_u2_or_zero(img, (size_t)(y7 + 1) * P.mv_w + x7, y7 + 1 < P.mv_h && x7 < P.mv_w);
    const uint2 d = ldg_u2_or_zero(img, (size_t)(y7 + 1) * P.mv_w + x7 + 1, y7 + 1 < P.mv_h && x7 + 1 < P.mv_w);
    L.t[0] = a.x; L.t[1] = a.y; L.t[2] = b.x; L.t[3] = b.y;
    L.t[4] = c.x; L.t[5] = c.y; L.t[6] = d.x; L.t[7] = d.y;
  }
  if (P.mode == LSFA_W_LOGITS || (P.mode == LSFA_W_COSINE && P.logits != nullptr)) {
    const float* l = P.logits + (size_t)n * 2 * P.HW;
    L.l0 = __ldg(l + p);
    L.l1 = __ldg(l + P.HW + p);
  }
  return L;
}

// Register-free first touch of everything issue_pixel_loads() will read: L2 prefetches for all of
// a thread's pixels go out back to back, so the loads that follow (one pixel at a time, because
// ptxas will not keep 10 words x PPT pixels live next to the hot loop's state) hit in L2.
__device__ __forceinline__ void prefetch_l2(const void* p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }

__device__ __forceinline__ void prefetch_pixel_loads(const AggParams& P, int n, int y, int x) {
  const int p = y * P.W + x;
  if (P.flow_kind == LSFA_FLOW_GRID || P.flow_kind == LSFA_FLOW_PREPOOLED) {
    const float* f = (const float*)P.flow + (size_t)n * 2 * P.HW;
    prefetch_l2(f + p);
    prefetch_l2(f + P.HW + p);
  } else if (P.pool_mode == LSFA_POOL_CENTRE2X2 && P.flow_kind != LSFA_FLOW_COVIAR_I32) {
    const char* img = (const char*)P.flow + (size_t)n * P.mv_h * P.mv_w * 8;
    const int y7 = 16 * y + 7, x7 = 16 * x + 7;   // x7 and x7+1 share a 32-byte sector unless x7*8 % 32 == 24
    if (y7 < P.mv_h && x7 < P.mv_w) prefetch_l2(img + ((size_t)y7 * P.mv_w + x7) * 8);
    if (y7 < P.mv_h && x7 + 1 < P.mv_w) prefetch_l2(img + ((size_t)y7 * P.mv_w + x7 + 1) * 8);
    if (y7 + 1 < P.mv_h && x7 < P.mv_w) prefetch_l2(img + ((size_t)(y7 + 1) * P.mv_w + x7) * 8);
    if (y7 + 1 < P.mv_h && x7 + 1 < P.mv_w) prefetch_l2(img + ((size_t)(y7 + 1) * P.mv_w + x7 + 1) * 8);
  }
  if (P.mode == LSFA_W_LOGITS || (P.mode == LSFA_W_COSINE && P.logits != nullptr)) {
    const float* l = P.logits + (size_t)n * 2 * P.HW;
    prefetch_l2(l + p);
    prefetch_l2(l + P.HW + p);
  }
}

__device__ __forceinline__ double raw_word(unsigned w, bool is_i32) {
  return is_i32 ? (double)(int)w : (double)__uint_as_float(w);
}

// Everything after the loads: a5/a6 pooling in float64, a7 grid, a8 index math, blend weights.
__device__ __forceinline__ PixelRec finish_pixel(const AggParams& P, const PixelLoads& L, int n, int y,
                                                 int x, bool fold = true) {
  float gx, gy;
  if (P.flow_kind == LSFA_FLOW_GRID) {
    gx = __uint_as_float(L.t[0]);
    gy = __uint_as_float(L.t[1]);
  } else {
    float fx, fy;
    if (P.flow_kind == LSFA_FLOW_PREPOOLED) {
      fx = __uint_as_float(L.t[0]);
      fy = __uint_as_float(L.t[1]);
    } else if (P.flow_kind == LSFA_FLOW_COVIAR_I32) {   // a1+a2 folded in: not prefetched (pre-pass / slow paths)
      const int* mv = (const int*)P.flow + (size_t)n * P.src_h * P.src_w * 2;
      fx = (float)__dmul_rn(coviar_pool_cell(P, mv, y, x, 0), P.mv_scale);
      fy = (float)__dmul_rn(coviar_pool_cell(P, mv, y, x, 1), P.mv_scale);
    } else if (P.pool_mode == LSFA_POOL_CENTRE2X2) {
      const bool i32 = P.flow_kind == LSFA_FLOW_RAW_I32;
      // ((a + b) + (c + d)) * 0.25 * (im_scale / 16), cv2's horizontal-pass-first order
      const double sx = __dmul_rn(__dadd_rn(__dadd_rn(raw_word(L.t[0], i32), raw_word(L.t[2], i32)),
                                            __dadd_rn(raw_word(L.t[4], i32), raw_word(L.t[6], i32))), 0.25);
      const double sy = __dmul_rn(__dadd_rn(__dadd_rn(raw_word(L.t[1], i32), raw_word(L.t[3], i32)),
                                            __dadd_rn(raw_word(L.t[5], i32), raw_word(L.t[7], i32))), 0.25);
      fx = (float)__dmul_rn(sx, P.mv_scale);
      fy = (float)__dmul_rn(sy, P.mv_scale);
    } else {  // avg16: 256 taps, not prefetched (not the parity mode)
      if (P.flow_kind == LSFA_FLOW_RAW_I32) {
        const int* mv = (const int*)P.flow + (size_t)n * P.mv_h * P.mv_w * 2;
        fx = (float)__dmul_rn(pool_cell(mv, P.mv_h, P.mv_w, 2, y, x, 0, P.pool_mode), P.mv_scale);
        fy = (float)__dmul_rn(pool_cell(mv, P.mv_h, P.mv_w, 2, y, x, 1, P.pool_mode), P.mv_scale);
      } else {
        const float* mv = (const float*)P.flow + (size_t)n * P.mv_h * P.mv_w * 2;
        fx = (float)__dmul_rn(pool_cell(mv, P.mv_h, P.mv_w, 2, y, x, 0, P.pool_mode), P.mv_scale);
        fy = (float)__dmul_rn(pool_cell(mv, P.mv_h, P.mv_w, 2, y, x, 1, P.pool_mode), P.mv_scale);
      }
    }
    gx = exact_grid(fx, (float)x, P.half_w);
    gy = exact_grid(fy, (float)y, P.half_h);
  }
  PixelRec t = make_taps(gx, gy, P.Hk, P.Wk, P.wk_m1, P.hk_m1);
  if (fold) {
    float ww = 1.0f, wc = 0.0f;
    if (P.mode == LSFA_W_ADD) {
      wc = 1.0f;
    } else if (P.mode == LSFA_W_MEAN) {
      ww = 0.5f;
      wc = 0.5f;
    } else if (P.mode == LSFA_W_LOGITS || P.mode == LSFA_W_COSINE) {
      softmax2(L.l0, L.l1, ww, wc);
    }
    fold_blend(t, ww, wc);
  }
  return t;
}

// Packed sampling record exchanged between the record pre-pass and the streaming kernel:
// two 16-byte words per output pixel.
__device__ __forceinline__ void pack_record(const PixelRec& t, uint4& a, uint4& b) {
  a = make_uint4(__float_as_uint(t.w00), __float_as_uint(t.w01), __float_as_uint(t.w10), __float_as_uint(t.w11));
  b = make_uint4(__float_as_uint(t.wc), __float_as_uint(t.ww),
                 (unsigned)(t.i00 * 4) | ((unsigned)(t.i01 * 4) << 16),
                 (unsigned)(t.i10 * 4) | ((unsigned)(t.i11 * 4) << 16));
}


// ---------------------------------------------------------------------------------------
// mbarrier + bulk async copy (global -> shared), SASS: SYNCS / UBLKCP
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return (uint32_t)__cvta_generic_to_shared(p);
}
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void fence_barrier_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)),
               "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred P1;\n"
      "LAB_WAIT:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1, %2;\n"
      "@P1 bra DONE;\n"
      "bra LAB_WAIT;\n"
      "DONE:\n"
      "}" ::"r"(smem_u32(bar)),
      "r"(parity), "r"(0x989680u)   // suspend-time hint (ns): sleep in hardware instead of spinning
      : "memory");
}
__device__ __forceinline__ void bulk_g2s(void* dst_smem, const void* src_gmem, uint32_t bytes,
                                         uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
      ::"r"(smem_u32(dst_smem)),
      "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
      : "memory");
}

// ---------------------------------------------------------------------------------------
// once-touched streams: bypass L1 allocation on load, streaming store
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ float ldg_stream(const float* p) {
  float v;
  asm volatile("ld.global.nc.L1::no_allocate.f32 %0, [%1];" : "=f"(v) : "l"(p));
  return v;
}
// Per-pixel sums a.a, b.b, a.b of the NCHW cosine (Fgfa_net compute_weight, SYM:111-116): the share of channel
// group grp (of kCosGroups; E/kCosGroups channels each, coalesced 128-byte rows) for pixel p < HW of frame n.  The
// caller adds the groups' sums in group order.  The forward (cosine_logits_nchw_kernel) and the backward's coefficient
// kernel both use it, so the backward recomputes the forward's bits.
constexpr int kCosGroups = 8;
__device__ __forceinline__ void cosine_group_sums_nchw(const float* __restrict__ ew, const float* __restrict__ ec, int E, int HW,
                                                       int n, int p, int grp, float& sww, float& scc, float& swc) {
  const size_t base = (size_t)n * E * HW + p;
  const int per = (E + kCosGroups - 1) / kCosGroups;
  const int e0 = grp * per, e1 = min(E, e0 + per);
  int e = e0;
  for (; e + 4 <= e1; e += 4) {
    float a[4], b[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      a[u] = ldg_stream(ew + base + (size_t)(e + u) * HW);
      b[u] = ldg_stream(ec + base + (size_t)(e + u) * HW);
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      sww = fmaf(a[u], a[u], sww);
      scc = fmaf(b[u], b[u], scc);
      swc = fmaf(a[u], b[u], swc);
    }
  }
  for (; e < e1; ++e) {
    const float a = ldg_stream(ew + base + (size_t)e * HW);
    const float b = ldg_stream(ec + base + (size_t)e * HW);
    sww = fmaf(a, a, sww);
    scc = fmaf(b, b, scc);
    swc = fmaf(a, b, swc);
  }
}

// Cache policy of the once-touched streams (compile-time experiment knob):
//   0: ld.global.nc.L1::no_allocate + st.global.cs   1: ld.global.nc (L1 allocate) + st.global.cs  <- default:
//      measured 5373 vs 4910 GB/s; the sector a warp shares with its neighbour then hits in L1
//   2: ld.global.nc.L1::no_allocate + st.global (write-back)   3: ld.global.nc + st.global
#ifndef LSFA_LD_POLICY
#define LSFA_LD_POLICY 1
#endif
#if (LSFA_LD_POLICY & 1)
#define LSFA_LD_STREAM "ld.global.nc.f32"
#else
#define LSFA_LD_STREAM "ld.global.nc.L1::no_allocate.f32"
#endif
#if (LSFA_LD_POLICY & 2)
#define LSFA_ST_STREAM "st.global.f32"
#else
#define LSFA_ST_STREAM "st.global.cs.f32"
#endif
// predicated forms: no branch, no load/store when ok == 0 (the result is then undefined)
__device__ __forceinline__ float ldg_stream_if(const float* p, unsigned ok) {
  float v;
  asm volatile(
      "{\n .reg .pred q;\n setp.ne.u32 q, %2, 0;\n mov.f32 %0, 0f00000000;\n"
      "@q " LSFA_LD_STREAM " %0, [%1];\n}"
      : "=f"(v)
      : "l"(p), "r"(ok));
  return v;
}
__device__ __forceinline__ void stg_stream_if(float* p, float v, unsigned ok) {
  asm volatile("{\n .reg .pred q;\n setp.ne.u32 q, %2, 0;\n @q " LSFA_ST_STREAM " [%0], %1;\n}" ::"l"(p), "f"(v),
               "r"(ok)
               : "memory");
}
__device__ __forceinline__ uint4 ldg_stream_v4(const void* p) {
  uint4 v;
  asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
               : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w)
               : "l"(p));
  return v;
}
__device__ __forceinline__ uint4 ldg_cached_v4(const void* p) {
  uint4 v;
  asm volatile("ld.global.nc.v4.u32 {%0,%1,%2,%3}, [%4];"
               : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w)
               : "l"(p));
  return v;
}
__device__ __forceinline__ void stg_stream(float* p, float v) {
  asm volatile("st.global.cs.f32 [%0], %1;" ::"l"(p), "f"(v) : "memory");
}
__device__ __forceinline__ void stg_stream_v4(void* p, uint4 v) {
  asm volatile("st.global.cs.v4.u32 [%0], {%1,%2,%3,%4};" ::"l"(p), "r"(v.x), "r"(v.y),
               "r"(v.z), "r"(v.w)
               : "memory");
}

// Packed dual-fp32 arithmetic (Blackwell FFMA2/FMUL2: one instruction, two IEEE fp32 results -
// bit-identical to two scalar fmaf/fmul).  A pair lives in a 64-bit register: lo = element 2i.
typedef unsigned long long f32x2;
__device__ __forceinline__ f32x2 pair2(float lo, float hi) {
  f32x2 d;
  asm("mov.b64 %0, {%1, %2};" : "=l"(d) : "f"(lo), "f"(hi));
  return d;
}
__device__ __forceinline__ void unpair2(f32x2 v, float& lo, float& hi) {
  asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ f32x2 fma2(f32x2 a, f32x2 b, f32x2 c) {
  f32x2 d;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
  return d;
}
__device__ __forceinline__ f32x2 mul2(f32x2 a, f32x2 b) {
  f32x2 d;
  asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
  return d;
}

// 16-byte vector <-> float lanes for the NHWC kernels
template <typename T>
struct Vec16;
template <>
struct Vec16<float> {
  static constexpr int kLanes = 4;
  __device__ static __forceinline__ void unpack(const uint4& v, float* f) {
    f[0] = __uint_as_float(v.x);
    f[1] = __uint_as_float(v.y);
    f[2] = __uint_as_float(v.z);
    f[3] = __uint_as_float(v.w);
  }
  __device__ static __forceinline__ uint4 pack(const float* f) {
    return make_uint4(__float_as_uint(f[0]), __float_as_uint(f[1]), __float_as_uint(f[2]),
                      __float_as_uint(f[3]));
  }
  // pair form: kLanes/2 packed f32x2
  __device__ static __forceinline__ void unpack2(const uint4& v, f32x2* f) {
    f[0] = pair2(__uint_as_float(v.x), __uint_as_float(v.y));
    f[1] = pair2(__uint_as_float(v.z), __uint_as_float(v.w));
  }
  __device__ static __forceinline__ uint4 pack2(const f32x2* f) {
    float a, b, c, d;
    unpair2(f[0], a, b);
    unpair2(f[1], c, d);
    return make_uint4(__float_as_uint(a), __float_as_uint(b), __float_as_uint(c), __float_as_uint(d));
  }
};
template <>
struct Vec16<__nv_bfloat16> {
  static constexpr int kLanes = 8;
  __device__ static __forceinline__ void unpack(const uint4& v, float* f) {
    const unsigned u[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int i = 0; i < 4; ++i) {  // bf16 -> f32 is a 16-bit shift
      f[2 * i] = __uint_as_float(u[i] << 16);
      f[2 * i + 1] = __uint_as_float(u[i] & 0xffff0000u);
    }
  }
  __device__ static __forceinline__ uint4 pack(const float* f) {
    unsigned u[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      __nv_bfloat162 h = __floats2bfloat162_rn(f[2 * i], f[2 * i + 1]);
      u[i] = *reinterpret_cast<unsigned*>(&h);
    }
    return make_uint4(u[0], u[1], u[2], u[3]);
  }
  __device__ static __forceinline__ void unpack2(const uint4& v, f32x2* f) {
    const unsigned u[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int i = 0; i < 4; ++i) f[i] = pair2(__uint_as_float(u[i] << 16), __uint_as_float(u[i] & 0xffff0000u));
  }
  __device__ static __forceinline__ uint4 pack2(const f32x2* f) {
    unsigned u[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      float lo, hi;
      unpair2(f[i], lo, hi);
      __nv_bfloat162 h = __floats2bfloat162_rn(lo, hi);
      u[i] = *reinterpret_cast<unsigned*>(&h);
    }
    return make_uint4(u[0], u[1], u[2], u[3]);
  }
};

}  // namespace lsfa
