// NCHW float32 path: host-side planning / dispatch of the plane-resident kernel
// (aggregate_nchw_plane.cuh, instantiated per variant in plane_var*.cu), the generic gather
// kernel for shapes the fast kernel does not take, and the cosine-logit pre-pass.
#include <cstdlib>

#include "aggregate_nchw_tma2.cuh"

namespace lsfa {

// ---------------------------------------------------------------------------------------
// Generic kernel: one thread per output pixel, CG channels per thread, taps gathered from
// global memory (L1/L2 serve the 4-tap reuse).  No alignment or size restriction.
// ---------------------------------------------------------------------------------------
constexpr int kGenericThreads = 256;
constexpr int kGenericCG = 16;

__global__ void __launch_bounds__(kGenericThreads)
agg_nchw_generic_kernel(const __grid_constant__ AggParams P) {
  const int n = blockIdx.z;
  const int p = blockIdx.x * kGenericThreads + threadIdx.x;
  if (p >= P.HW) return;
  const int c_begin = blockIdx.y * kGenericCG;
  const int c_end = min(P.C, c_begin + kGenericCG);
  const float* __restrict__ scale = static_cast<const float*>(P.scale);
  const float* __restrict__ cur = static_cast<const float*>(P.cur);
  float* __restrict__ out = static_cast<float*>(P.out);
  const bool has_cur = P.mode != LSFA_W_NONE;
  const bool byp = (P.bypass != nullptr) && (__ldg(P.bypass + n) != 0);

  if (byp) {
    for (int c = c_begin; c < c_end; ++c) {
      const size_t e = ((size_t)n * P.C + c) * P.HW + p;
      float o = cur[e];
      if (P.req_add) o += out[e];
      out[e] = o;
    }
    return;
  }
  const int y = p / P.W, x = p - y * P.W;
  const PixelLoads ld = issue_pixel_loads(P, n, y, x);
  const PixelRec t = finish_pixel(P, ld, n, y, x);
  float r0 = 0.f, r1 = 0.f, r2 = 0.f;
  if (P.res) {
    r0 = __ldg(P.res + ((size_t)n * 3 + 0) * P.HW + p);
    r1 = __ldg(P.res + ((size_t)n * 3 + 1) * P.HW + p);
    r2 = __ldg(P.res + ((size_t)n * 3 + 2) * P.HW + p);
  }
  const int kn = key_slot(P, n);
  for (int c = c_begin; c < c_end; ++c) {
    const float* __restrict__ plane = static_cast<const float*>(P.key) + ((size_t)kn * P.C + c) * P.HWk;
    const size_t e = ((size_t)n * P.C + c) * P.HW + p;
    float v = tap_chain(t, __ldg(plane + t.i00), __ldg(plane + t.i01), __ldg(plane + t.i10), __ldg(plane + t.i11));
    if (scale) v *= __ldg(scale + e);
    if (P.res)
      v = fmaf(t.ww, rnet_term(__ldg(P.rnet_w + (size_t)c * 3), __ldg(P.rnet_w + (size_t)c * 3 + 1),
                               __ldg(P.rnet_w + (size_t)c * 3 + 2), __ldg(P.rnet_b + c), r0, r1, r2), v);
    float o = has_cur ? fmaf(t.wc, __ldg(cur + e), v) : v;
    if (P.req_add) o += out[e];
    out[e] = o;
  }
}

// ---------------------------------------------------------------------------------------
// Cosine logits from NCHW embeddings (Fgfa_net compute_weight, SYM:111-116,137-139).
// Block = 32 pixels x 8 channel groups (cosine_group_sums_nchw); the groups' partial sums are
// combined in a fixed order in shared memory.
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(32 * kCosGroups)
cosine_logits_nchw_kernel(const float* __restrict__ ew, const float* __restrict__ ec,
                          float* __restrict__ logits, int E, int HW) {
  __shared__ float part[3][kCosGroups][32];
  const int n = blockIdx.y;
  const int lane = threadIdx.x & 31, grp = threadIdx.x >> 5;
  const int p = blockIdx.x * 32 + lane;
  float sww = 0.f, scc = 0.f, swc = 0.f;
  if (p < HW) cosine_group_sums_nchw(ew, ec, E, HW, n, p, grp, sww, scc, swc);
  part[0][grp][lane] = sww;
  part[1][grp][lane] = scc;
  part[2][grp][lane] = swc;
  __syncthreads();
  if (grp == 0 && p < HW) {
    float tww = 0.f, tcc = 0.f, twc = 0.f;
#pragma unroll
    for (int g = 0; g < kCosGroups; ++g) {
      tww += part[0][g][lane];
      tcc += part[1][g][lane];
      twc += part[2][g][lane];
    }
    const float nw = sqrtf(tww + 1e-10f), nc = sqrtf(tcc + 1e-10f);
    logits[((size_t)n * 2 + 0) * HW + p] = twc / (nw * nc);
    logits[((size_t)n * 2 + 1) * HW + p] = tcc / (nc * nc);
  }
}

// ---------------------------------------------------------------------------------------
// host-side launchers
// ---------------------------------------------------------------------------------------
static int g_sm_count_cache[64];  // written once per device with the same value: benign

static int sm_count() {
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return 148;
  if (dev >= 0 && dev < 64 && g_sm_count_cache[dev] > 0) return g_sm_count_cache[dev];
  int n = 148;
  cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
  if (dev >= 0 && dev < 64) g_sm_count_cache[dev] = n;
  return n;
}

// Decide whether the plane-resident kernel can serve these args; fill the tiling fields.
bool plan_plane_kernel(AggParams& P, size_t* smem_out) {
  const size_t kSmemBudget = 220 * 1024;
  if (P.HW > 8 * kPlaneThreads * 64) return false;
  if (P.HWk > 16383) return false;                     // tap byte offsets are packed in 16 bits
  int K = 0;
  const int prefer[2] = {2, 4};
  for (int i = 0; i < 2 && K == 0; ++i) {
    const int k = prefer[i];
    if (P.C % k) continue;
    if (((long long)k * P.HWk) % 4) continue;          // bulk copy size multiple of 16 B
    if ((size_t)k * P.HWk * 4 > 96 * 1024) continue;   // keep >= 2 stages
    K = k;
  }
  if (K == 0) return false;
  if (reinterpret_cast<uintptr_t>(P.key) % 16) return false;
  if (((long long)P.C * P.HWk) % 4) return false;      // every frame's planes stay 16 B aligned
  // pixel slots per thread: 8 only for the lean variants at K=2 (register budget), else <= 5
  const bool lean = !P.req_add && P.res == nullptr;
  const int n_opt = (K == 2 && lean) ? 4 : 3;
  const int ppt_options[4] = {1, 3, 5, 8};
  int ppt = ppt_options[n_opt - 1];
  for (int i = n_opt - 1; i >= 0; --i)
    if ((long long)ppt_options[i] * kPlaneThreads >= P.HW) ppt = ppt_options[i];
  P.K = K;
  P.chunks = P.C / K;
  P.part_pix = ppt * kPlaneThreads;
  P.parts = (P.HW + P.part_pix - 1) / P.part_pix;
  P.stage_bytes = (unsigned)((size_t)K * P.HWk * 4);
  const size_t res_bytes = P.res ? (size_t)3 * P.part_pix * 4 : 0;
  long long stages = ((long long)kSmemBudget - kBarrierBytes - (long long)res_bytes) / P.stage_bytes;
  if (stages < 2) return false;
  if (stages > kMaxStages) stages = kMaxStages;
  P.stages = (int)stages;
  P.items = (long long)P.N * P.chunks * P.parts;
  *smem_out = kBarrierBytes + (size_t)P.stages * P.stage_bytes + res_bytes;
  return true;
}

cudaError_t launch_agg_nchw_plane(const AggParams& P, size_t smem, cudaStream_t st) {
  long long grid = sm_count();
  if (grid > P.items) grid = P.items;
  const bool has_scale = P.scale != nullptr, has_cur = P.mode != LSFA_W_NONE, has_res = P.res != nullptr;
  // this kernel is the fallback of the all-TMA one: only the run-time-flag form and the key-frame
  // blend (kept specialised for the LDG/STG-vs-TMA ablation) are instantiated
  if (!P.req_add && has_scale && has_cur && !has_res) return launch_plane_variant<kVarScaleCur>(P, smem, (int)grid, st);
  (void)has_res;
  return launch_plane_variant<kVarRuntime>(P, smem, (int)grid, st);
}

// ---------------------------------------------------------------------------------------
// Record pre-pass: every index-math row of the path (a3,a5,a6 MV pooling in float64, a7 grid,
// a8 floor/weights, a13 softmax, blend fold) once per output pixel, written as a 32-byte packed
// record.  The streaming kernel then rebuilds its per-frame state with two 16-byte loads per
// pixel instead of redoing this math in every CTA that touches the frame (the sparse raw-MV
// taps cost ~10 us of LSU time per rebuild: -8% on the fused kernel when done in place).
// It runs just before the streaming kernel in stream order (~3 us for 64 frames).
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) agg_records_kernel(const __grid_constant__ AggParams P, uint4* __restrict__ rec) {
  const long long total = (long long)P.N * P.HW;
  if (P.zero_counter != nullptr && blockIdx.x == 0 && threadIdx.x == 0) *P.zero_counter = 0u;   // the kernel that claims from it follows in stream order
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const int n = (int)(i / P.HW);
    const int p = (int)(i - (long long)n * P.HW);
    if (P.bypass != nullptr && __ldg(P.bypass + n) != 0) continue;   // never read for bypass frames
    const int y = p / P.W, x = p - y * P.W;
    const PixelLoads ld = issue_pixel_loads(P, n, y, x);
    PixelRec t = finish_pixel(P, ld, n, y, x);
    if (P.canon) canonical_taps(t, P.Hk, P.Wk);
    uint4 a, b;
    pack_record(t, a, b);
    rec[2 * i] = a;
    rec[2 * i + 1] = b;
    if (P.rowrange != nullptr) {
      // key rows this pixel's (clamped) taps read: the streaming kernel loads only the rows its part needs
      const int vf = n * P.parts + p / P.part_pix;
      unsigned hi = (unsigned)(t.i10 / P.Wk) + 1u, lo_inv = (unsigned)(P.Hk - t.i00 / P.Wk);
      const unsigned act = __activemask();
      const int vf0 = __shfl_sync(act, vf, __ffs(act) - 1);
      if (__all_sync(act, vf == vf0)) {          // the usual case: one atomic pair per warp
        hi = __reduce_max_sync(act, hi);
        lo_inv = __reduce_max_sync(act, lo_inv);
        if ((threadIdx.x & 31) == __ffs(act) - 1) {
          atomicMax(P.rowrange + 2 * vf, hi);
          atomicMax(P.rowrange + 2 * vf + 1, lo_inv);
        }
      } else {
        atomicMax(P.rowrange + 2 * vf, hi);
        atomicMax(P.rowrange + 2 * vf + 1, lo_inv);
      }
    }
  }
}

cudaError_t launch_agg_records(const AggParams& P, uint4* rec, cudaStream_t st) {
  const long long total = (long long)P.N * P.HW;
  long long grid = (total + 255) / 256;
  if (grid > 148LL * 8) grid = 148LL * 8;
  agg_records_kernel<<<(unsigned)grid, 256, 0, st>>>(P, rec);
  return cudaPeekAtLastError();
}

// ---- all-TMA kernel: planning and dispatch -------------------------------------------------
static int variant_of(const AggParams& P) {
  const bool has_scale = P.scale != nullptr, has_cur = P.mode != LSFA_W_NONE, has_res = P.res != nullptr;
  if (P.req_add) return kVarRuntime;
  if (!has_scale && !has_cur && !has_res) return kVarWarpOnly;
  if (has_scale && !has_cur && !has_res) return kVarScale;
  if (has_scale && has_cur && !has_res) return kVarScaleCur;
  if (!has_scale && has_cur && has_res) return kVarResCur;
  return kVarRuntime;
}

bool plan_tma_kernel(AggParams& P, size_t* smem_out) {
  const size_t kSmemMax = 227 * 1024;
  const int var = variant_of(P);
  if (var == kVarRuntime) return false;
  if (P.HWk > 16383) return false;                               // tap byte offsets are packed in 16 bits
  if (var == kVarWarpOnly && (P.Hk < 2 || P.Wk < 2)) return false;   // canonical_taps(): a 2x2 block inside the plane
  const void* ptrs[4] = {P.key, P.scale, P.cur, P.out};
  for (const void* q : ptrs)
    if (q && (reinterpret_cast<uintptr_t>(q) % 16)) return false;
  if (((long long)P.C * P.HW) % 4 || ((long long)P.C * P.HWk) % 4) return false;
  // pixel slots per consumer thread; planes beyond 9*480 pixels are cut into balanced parts,
  // which needs every plane slice 16-byte aligned (HW % 4 == 0)
  const int ppt_options[4] = {1, 3, 5, 9};
  const int max_part = 9 * kTmaConsumers;
  const int parts = (P.HW + max_part - 1) / max_part;
  if (parts > 1 && (P.HW % 4)) return false;
  const int per_part = (P.HW + parts - 1) / parts;
  int ppt = 9;
  for (int i = 3; i >= 0; --i)
    if ((long long)ppt_options[i] * kTmaConsumers >= per_part) ppt = ppt_options[i];
  const int part_pix = ppt * kTmaConsumers;
  if ((long long)part_pix * (parts - 1) >= P.HW) return false;   // every part must be non-empty
  const bool has_scale = var == kVarScale || var == kVarScaleCur;
  // res variant: pooled residual of the frame part [3][part_pix] + the rnet_conv0 table [C] x (w0,w1,w2,b)
  // (up to 5 pixel slots per thread keep the residual in registers: no [3][part_pix] array)
  const size_t res_bytes = var == kVarResCur ? (ppt <= 5 ? 0 : (size_t)3 * part_pix * 4) + (size_t)P.C * 16 : 0;
  const int io_plane = parts == 1 ? P.HW : part_pix;             // elements per plane slice in a stage
  const size_t pad = (((size_t)part_pix - (parts == 1 ? P.HW : 0)) * 4 + 127) / 128 * 128;
  const int prefer[2] = {2, 1};   // (four planes per item measured slower on the warp-only variant: 0.79 -> 0.74)
  for (int i = 0; i < 2; ++i) {
    const int K = prefer[i];
    if (P.C % K) continue;
    if (((long long)K * P.HW) % 4 || ((long long)K * P.HWk) % 4) continue;   // 16-byte bulk copies
    const unsigned key_bytes = (unsigned)((size_t)K * P.HWk * 4), io_bytes = (unsigned)((size_t)K * io_plane * 4);
    const unsigned off_scale = (key_bytes + 127u) / 128u * 128u;
    const unsigned off_io = has_scale ? off_scale + (io_bytes + 127u) / 128u * 128u : off_scale;
    // warp-only variant: the consumers store straight to global (measured 6-8 % faster: this variant is bound by
    // shared-memory bandwidth, and the staged form costs one STS plus one copy-engine read per element), so its
    // stages hold key planes only.
    const bool direct = var == kVarWarpOnly;                     // compile-time in the kernel (tma_consumer_loop<.., DIRECT>)
    const unsigned stage_bytes = direct ? off_scale : off_io + (io_bytes + 127u) / 128u * 128u;
    // (variants WITH a current feature keep the staged store: direct stores measured 168.2k -> 167.4k frames/s on the
    // headline and 167k -> 133k on the shared-key stream sweep, round 2)
    P.direct_store = direct ? 1 : 0;
    long long stages = ((long long)kSmemMax - kTmaHeaderBytes - (long long)res_bytes - (long long)pad) / stage_bytes;
    if (stages > kMaxStages) stages = kMaxStages;
    if (stages < 3 && !(K == 1 && stages >= 2)) continue;    // want >= 3 stages; K=1 may run with 2
    P.K = K;
    P.chunks = P.C / K;
    P.parts = parts;
    P.part_pix = part_pix;
    P.stages = (int)stages;
    P.stage_bytes = stage_bytes;
    P.key_bytes = key_bytes;
    P.io_bytes = io_bytes;
    P.off_scale = off_scale;
    P.off_io = off_io;
    P.items = (long long)P.N * parts * P.chunks;
    *smem_out = kTmaHeaderBytes + (size_t)P.stages * stage_bytes + res_bytes + pad;
    return true;
  }
  return false;
}

cudaError_t launch_agg_nchw_tma(const AggParams& Pin, size_t smem, cudaStream_t st) {
  AggParams P = Pin;
  P.canon = variant_of(P) == kVarWarpOnly ? 1 : 0;          // canonical tap records: see tma_consumer_loop
  if (knob("LSFA_TMA_STATIC")) P.sched = nullptr;          // experiment knobs (ablations)
  if (knob("LSFA_TMA_NO_RECORDS")) P.records = nullptr;
  {
    // share of the items handed out dynamically at the end (the rest is a static contiguous split)
    int pct = kTmaPoolPercent;
    if (const char* e = knob("LSFA_TMA_POOL_PCT")) pct = atoi(e);
    if (pct < 0) pct = 0;
    if (pct > 100) pct = 100;
    P.pool_base = P.items - P.items * pct / 100;
    P.pool_base -= P.pool_base % kTmaClaim;                  // claims stay aligned to the claim size
  }
  long long grid = sm_count();
  if (grid > P.items) grid = P.items;
  // planes cut into pixel parts: each part loads only the key rows its taps read (found by the pre-pass);
  // needs whole rows / planes to stay 16-byte addressable
  const bool trim = P.sched && P.records && !P.records_ready && P.parts > 1 && (P.HWk % 4) == 0 && knob("LSFA_NO_ROW_TRIM") == nullptr;
  P.rowrange = trim ? P.sched + (size_t)P.N * P.parts : nullptr;
  // small batches (the reference's batch-1 operating mode, BASELINE configs[0]): ONE cooperative launch - the kernel's own
  // consumers build the records before a grid-wide barrier; static work split, whole key planes: no pre-pass, no memset
  P.coop = (P.records != nullptr && !P.records_ready && (long long)P.N * P.parts <= kCoopMaxVirtualFrames &&
            knob("LSFA_TMA_NO_COOP") == nullptr) ? 1 : 0;
  if (P.coop) {
    P.sched = nullptr;
    P.rowrange = nullptr;
    P.pool_base = P.items;
  }
  // the claim counter (and, row-trimmed, the row ranges the pre-pass reduces into) start every launch at zero; without row
  // ranges the pre-pass zeroes the one counter itself: one graph node less per step (~2-3 us of 378 on the headline)
  const bool prepass = P.records && !P.coop && !P.records_ready;
  if (P.sched && (trim || !prepass)) {
    cudaError_t e = cudaMemsetAsync(P.sched, 0, (size_t)P.N * P.parts * sizeof(unsigned) * (trim ? 3 : 1), st);
    if (e != cudaSuccess) return e;
  }
  if (prepass) {  // pre-pass writes the records, the streaming kernel follows in stream order
    AggParams R = P;
    R.records = nullptr;
    R.zero_counter = (P.sched && !trim) ? P.sched : nullptr;
    cudaError_t e = launch_agg_records(R, const_cast<uint4*>(P.records), st);
    if (e != cudaSuccess) return e;
  }
  switch (variant_of(P)) {
    case kVarWarpOnly: return launch_tma_variant<kVarWarpOnly>(P, smem, (int)grid, st);
    case kVarScale: return launch_tma_variant<kVarScale>(P, smem, (int)grid, st);
    case kVarScaleCur: return launch_tma_variant<kVarScaleCur>(P, smem, (int)grid, st);
    case kVarResCur: return launch_tma_variant<kVarResCur>(P, smem, (int)grid, st);
    default: return cudaErrorInvalidValue;
  }
}

// ---- 2-CTA cluster kernel (planes that need exactly two pixel parts): planning and dispatch ----
bool plan_tma2_kernel(AggParams& P, size_t* smem_out, bool forced) {
  (void)forced;
  const size_t kSmemMax = 227 * 1024;
  const int var = variant_of(P);
  if (var == kVarRuntime) return false;
  if (P.HWk > 16383 || (P.HW % 4) || (P.HWk % 4)) return false;
  const void* ptrs[4] = {P.key, P.scale, P.cur, P.out};
  for (const void* q : ptrs)
    if (q && (reinterpret_cast<uintptr_t>(q) % 16)) return false;
  const int per_part = (P.HW + 1) / 2;
  int ppt = 0;
  if (per_part > 5 * kTmaConsumers && per_part <= 9 * kTmaConsumers) ppt = 9;
  else if (per_part > 3 * kTmaConsumers && per_part <= 5 * kTmaConsumers) ppt = 5;
  if (ppt == 0) return false;                                   // one part fits a single CTA, or more than two are needed
  const int part_pix = ppt * kTmaConsumers;
  if (part_pix >= P.HW) return false;
  if (sm_count() < 2) return false;
  const bool has_scale = var == kVarScale || var == kVarScaleCur;
  const size_t res_bytes = var == kVarResCur ? (ppt <= 5 ? 0 : (size_t)3 * part_pix * 4) + (size_t)P.C * 16 : 0;
  const int K = 1;
  const unsigned key_bytes = (unsigned)((size_t)K * P.HWk * 4), io_bytes = (unsigned)((size_t)K * part_pix * 4);
  const unsigned off_scale = (key_bytes + 127u) / 128u * 128u;
  const unsigned off_io = has_scale ? off_scale + (io_bytes + 127u) / 128u * 128u : off_scale;
  const unsigned stage_bytes = off_io + (io_bytes + 127u) / 128u * 128u;
  long long stages = ((long long)kSmemMax - kTma2HeaderBytes - (long long)res_bytes) / stage_bytes;
  if (stages > kMaxStages) stages = kMaxStages;
  if (stages < 3) return false;
  P.K = K;
  P.chunks = P.C / K;
  P.parts = 2;
  P.part_pix = part_pix;
  P.stages = (int)stages;
  P.stage_bytes = stage_bytes;
  P.key_bytes = key_bytes;
  P.io_bytes = io_bytes;
  P.off_scale = off_scale;
  P.off_io = off_io;
  P.items = (long long)P.N * P.chunks;                          // one item = both parts of a (frame, chunk)
  *smem_out = kTma2HeaderBytes + (size_t)P.stages * stage_bytes + res_bytes;
  return true;
}

cudaError_t launch_agg_nchw_tma2(const AggParams& Pin, size_t smem, cudaStream_t st) {
  AggParams P = Pin;
  long long clusters = sm_count() / 2;
  if (clusters > P.items) clusters = P.items;
  if (P.sched) {
    cudaError_t e = cudaMemsetAsync(P.sched, 0, (size_t)P.N * sizeof(unsigned), st);
    if (e != cudaSuccess) return e;
  }
  if (P.records) {
    AggParams R = P;
    R.records = nullptr;
    cudaError_t e = launch_agg_records(R, const_cast<uint4*>(P.records), st);
    if (e != cudaSuccess) return e;
  }
  P.coop = 0;
  const int grid = (int)clusters * 2;
  switch (variant_of(P)) {
    case kVarWarpOnly: return launch_tma2_variant<kVarWarpOnly>(P, smem, grid, st);
    case kVarScale: return launch_tma2_variant<kVarScale>(P, smem, grid, st);
    case kVarScaleCur: return launch_tma2_variant<kVarScaleCur>(P, smem, grid, st);
    case kVarResCur: return launch_tma2_variant<kVarResCur>(P, smem, grid, st);
    default: return cudaErrorInvalidValue;
  }
}

cudaError_t launch_agg_nchw_generic(const AggParams& P, cudaStream_t st) {
  dim3 grid((P.HW + kGenericThreads - 1) / kGenericThreads, (P.C + kGenericCG - 1) / kGenericCG, P.N);
  if (grid.y > 65535 || grid.z > 65535) return cudaErrorInvalidValue;
  agg_nchw_generic_kernel<<<grid, kGenericThreads, 0, st>>>(P);
  return cudaPeekAtLastError();
}

cudaError_t launch_cosine_logits_nchw(const float* ew, const float* ec, float* logits, int N,
                                      int E, int HW, cudaStream_t st) {
  dim3 grid((HW + 31) / 32, N);
  if (grid.y > 65535) return cudaErrorInvalidValue;
  cosine_logits_nchw_kernel<<<grid, 32 * kCosGroups, 0, st>>>(ew, ec, logits, E, HW);
  return cudaPeekAtLastError();
}

}  // namespace lsfa
