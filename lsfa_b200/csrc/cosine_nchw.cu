// Cosine logits of Fgfa_net from NCHW (channel-planar) embeddings, all-TMA form.
//   compute_weight SYM:111-116: l = sum_c l2n(a)_c * l2n(b)_c, L2Normalization(mode='channel', eps 1e-10);
//   Fgfa_net SYM:137-139: logits[n,0] = cos(emb_warp, emb_cur), logits[n,1] = cos(emb_cur, emb_cur).
// This is the largest stream of the cosine variant (2 x 2048 x HW floats per frame, twice the four feature
// tensors together), so it gets the same treatment as the fused kernel: a producer lane moves whole channel
// planes HBM -> smem with cp.async.bulk (each byte once, no sector over-fetch on the 8-byte-phase planes), 15
// consumer warps keep three running sums (a.a, b.b, a.b) per owned pixel in registers.
// Work = (frame, pair of channels), split statically and contiguously over the CTAs; a CTA writes ONE partial
// per frame it touches into a fixed slot (slot = its rank among the CTAs touching that frame), and a second tiny
// kernel adds the slots in order: the sums are deterministic (no float atomics).
#include "aggregate_nchw_tma.cuh"

namespace lsfa {

struct CosParams {
  const float* ew;
  const float* ec;
  float* part;        // [N][slots][3][HW]
  float* logits;      // [N][2][HW]
  int N, E, HW, chunks, slots, stages;
  unsigned pair_bytes, stage_bytes;
  long long items;
};

// CTA whose static range [items*b/grid, items*(b+1)/grid) contains item i
__host__ __device__ inline int cos_owner(long long i, long long items, int grid) {
  int g = (int)((i * grid) / items);
  while (g > 0 && items * g / grid > i) --g;
  while (g + 1 < grid && items * (g + 1) / grid <= i) ++g;
  return g;
}

template <int PPT>
__global__ void __launch_bounds__(kTmaThreads, 1) cosine_partials_tma_kernel(const __grid_constant__ CosParams P) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  uint64_t* full = reinterpret_cast<uint64_t*>(smem_raw);
  uint64_t* empty = full + kMaxStages;
  unsigned char* ring = smem_raw + kTmaHeaderBytes;
  const int tid = threadIdx.x, warp = tid >> 5;
  const long long i0 = P.items * (long long)blockIdx.x / gridDim.x, i1 = P.items * (long long)(blockIdx.x + 1) / gridDim.x;
  if (tid == 0) {
    for (int s = 0; s < P.stages; ++s) {
      mbar_init(&full[s], 1);
      mbar_init(&empty[s], kTmaConsumerWarps);
    }
    fence_barrier_init();
  }
  __syncthreads();

  if (warp == kTmaConsumerWarps) {
    if ((tid & 31) == 0) {
      int s = 0;
      unsigned ph = 0;
      for (long long i = i0; i < i1; ++i) {
        if (i - i0 >= P.stages) mbar_wait(&empty[s], ph ^ 1u);     // the stage's previous occupant has been consumed
        unsigned char* st = ring + (size_t)s * P.stage_bytes;
        const size_t off = (size_t)i * 2 * P.HW;                   // item i = (n, pair): planes are contiguous over (n, e)
        mbar_expect_tx(&full[s], 2u * P.pair_bytes);
        bulk_g2s(st, P.ew + off, P.pair_bytes, &full[s]);
        bulk_g2s(st + P.stage_bytes / 2, P.ec + off, P.pair_bytes, &full[s]);
        if (++s == P.stages) {
          s = 0;
          ph ^= 1u;
        }
      }
    }
    return;
  }

  float sww[PPT], scc[PPT], swc[PPT];
#pragma unroll
  for (int j = 0; j < PPT; ++j) sww[j] = scc[j] = swc[j] = 0.f;
  auto flush = [&](int n) {
    const int slot = (int)blockIdx.x - cos_owner((long long)n * P.chunks, P.items, (int)gridDim.x);
    float* dst = P.part + ((size_t)n * P.slots + slot) * 3 * P.HW;
#pragma unroll
    for (int j = 0; j < PPT; ++j) {
      const int p = tid + j * kTmaConsumers;
      if (p < P.HW) {
        dst[p] = sww[j];
        dst[P.HW + p] = scc[j];
        dst[2 * P.HW + p] = swc[j];
      }
      sww[j] = scc[j] = swc[j] = 0.f;
    }
  };
  int s = 0, cur_n = -1;
  unsigned ph = 0;
  for (long long i = i0; i < i1; ++i) {
    const int n = (int)(i / P.chunks);
    if (n != cur_n) {
      if (cur_n >= 0) flush(cur_n);
      cur_n = n;
    }
    mbar_wait(&full[s], ph);
    const float* a_s = reinterpret_cast<const float*>(ring + (size_t)s * P.stage_bytes);
    const float* b_s = reinterpret_cast<const float*>(ring + (size_t)s * P.stage_bytes + P.stage_bytes / 2);
#pragma unroll
    for (int k = 0; k < 2; ++k) {
      float a[PPT], b[PPT];
#pragma unroll
      for (int j = 0; j < PPT; ++j) {
        const int p = tid + j * kTmaConsumers;
        const bool ok = p < P.HW;
        a[j] = ok ? a_s[k * P.HW + p] : 0.f;
        b[j] = ok ? b_s[k * P.HW + p] : 0.f;
      }
#pragma unroll
      for (int j = 0; j < PPT; ++j) {
        sww[j] = fmaf(a[j], a[j], sww[j]);
        scc[j] = fmaf(b[j], b[j], scc[j]);
        swc[j] = fmaf(a[j], b[j], swc[j]);
      }
    }
    __syncwarp();
    if ((tid & 31) == 0) mbar_arrive(&empty[s]);
    if (++s == P.stages) {
      s = 0;
      ph ^= 1u;
    }
  }
  if (cur_n >= 0) flush(cur_n);
}

// add the per-CTA partials of every frame in slot order, then the two cosines
__global__ void __launch_bounds__(256) cosine_finalize_kernel(const __grid_constant__ CosParams P, int grid_main) {
  const long long total = (long long)P.N * P.HW;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int n = (int)(i / P.HW), p = (int)(i - (long long)n * P.HW);
    const int first = cos_owner((long long)n * P.chunks, P.items, grid_main);
    const int last = cos_owner((long long)n * P.chunks + P.chunks - 1, P.items, grid_main);
    float tww = 0.f, tcc = 0.f, twc = 0.f;
    for (int j = 0; j <= last - first; ++j) {
      const float* src = P.part + ((size_t)n * P.slots + j) * 3 * P.HW;
      tww += src[p];
      tcc += src[P.HW + p];
      twc += src[2 * P.HW + p];
    }
    const float nw = sqrtf(tww + 1e-10f), nc = sqrtf(tcc + 1e-10f);
    P.logits[((size_t)n * 2 + 0) * P.HW + p] = twc / (nw * nc);
    P.logits[((size_t)n * 2 + 1) * P.HW + p] = tcc / (nc * nc);
  }
}

static int cos_sm_count() {
  int dev = 0, n = 148;
  if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
  return n > 0 ? n : 148;
}

static bool plan_cosine_tma(const float* ew, const float* ec, int N, int E, int HW, CosParams& P, int* grid, size_t* smem,
                            int* ppt) {
  if (E % 2 || (2LL * HW) % 4 || HW > 9 * kTmaConsumers) return false;
  if ((reinterpret_cast<uintptr_t>(ew) % 16) || (reinterpret_cast<uintptr_t>(ec) % 16)) return false;
  P.ew = ew; P.ec = ec; P.N = N; P.E = E; P.HW = HW;
  P.chunks = E / 2;
  P.items = (long long)N * P.chunks;
  P.pair_bytes = (unsigned)(2u * HW * 4u);
  P.stage_bytes = 2u * ((P.pair_bytes + 127u) / 128u * 128u);
  long long st = (227 * 1024 - kTmaHeaderBytes) / P.stage_bytes;
  if (st > kMaxStages) st = kMaxStages;
  if (st < 2) return false;
  P.stages = (int)st;
  long long g = cos_sm_count();
  if (g > P.items) g = P.items;
  *grid = (int)g;
  int slots = 1;
  for (int n = 0; n < N; ++n) {
    const int c = cos_owner((long long)n * P.chunks + P.chunks - 1, P.items, (int)g) - cos_owner((long long)n * P.chunks, P.items, (int)g) + 1;
    if (c > slots) slots = c;
  }
  P.slots = slots;
  *smem = kTmaHeaderBytes + (size_t)P.stages * P.stage_bytes;
  *ppt = HW <= 5 * kTmaConsumers ? 5 : 9;
  return true;
}

// scratch the TMA form needs for its partial sums (0 = it cannot serve these arguments)
size_t cosine_tma_workspace_bytes(int N, int E, int HW) {
  CosParams P;
  int grid = 0, ppt = 0;
  size_t smem = 0;
  if (!plan_cosine_tma(reinterpret_cast<const float*>(16), reinterpret_cast<const float*>(16), N, E, HW, P, &grid, &smem, &ppt))
    return 0;
  // the grid depends on the SM count of the current device; size for the worst case (one slot per CTA of a 148+ SM part)
  const size_t slots = (size_t)P.slots > 4 ? (size_t)P.slots : 4;
  return (size_t)N * slots * 3 * HW * sizeof(float);
}

// returns cudaErrorNotSupported when the arguments / scratch do not fit: the caller then runs the LDG kernel
cudaError_t launch_cosine_logits_nchw_tma(const float* ew, const float* ec, float* logits, int N, int E, int HW,
                                          void* scratch, size_t scratch_bytes, cudaStream_t st) {
  CosParams P;
  int grid = 0, ppt = 0;
  size_t smem = 0;
  if (!scratch || (reinterpret_cast<uintptr_t>(scratch) % 16)) return cudaErrorNotSupported;
  if (!plan_cosine_tma(ew, ec, N, E, HW, P, &grid, &smem, &ppt)) return cudaErrorNotSupported;
  if (scratch_bytes < (size_t)N * P.slots * 3 * HW * sizeof(float)) return cudaErrorNotSupported;
  P.part = static_cast<float*>(scratch);
  P.logits = logits;
  cudaError_t e;
  if (ppt == 5) {
    e = cudaFuncSetAttribute(cosine_partials_tma_kernel<5>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    cosine_partials_tma_kernel<5><<<grid, kTmaThreads, smem, st>>>(P);
  } else {
    e = cudaFuncSetAttribute(cosine_partials_tma_kernel<9>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    cosine_partials_tma_kernel<9><<<grid, kTmaThreads, smem, st>>>(P);
  }
  e = cudaPeekAtLastError();
  if (e != cudaSuccess) return e;
  const long long total = (long long)N * HW;
  long long fg = (total + 255) / 256;
  if (fg > 148 * 8) fg = 148 * 8;
  cosine_finalize_kernel<<<(unsigned)fg, 256, 0, st>>>(P, grid);
  return cudaPeekAtLastError();
}

// ---------------------------------------------------------------------------------------------------------------------
// Backward of the cosine logits (NCHW float32).  Per frame n and pixel p, with a = emb_warp[n,:,p], b = emb_cur[n,:,p],
// the forward's sums Saa, Sbb, Sab, na = sqrtf(Saa + 1e-10f), nb = sqrtf(Sbb + 1e-10f), l1 = Sab/(na nb), l2 = Sbb/(nb nb)
// and g1, g2 = d/d(l1), d/d(l2):
//   alpha = g1/(na nb),  beta = -g1 l1/na^2,  gamma = (-g1 l1 + 2 g2 (1 - l2))/nb^2
//   grad_emb_warp[c] = alpha b_c + beta a_c,   grad_emb_cur[c] = alpha a_c + gamma b_c
// Pass 1 recomputes the sums with the forward's own kernel and summation order (so l1, l2 are the forward's bits) and
// writes (alpha, beta, gamma) per pixel; pass 2 streams both embeddings once and writes both gradients.  Both gradient
// kernels evaluate the same two fmaf expressions, so they agree bit for bit.
// ---------------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void cosine_coefficients(float tww, float tcc, float twc, float g1, float g2, float& al, float& be,
                                                    float& ga) {
  const float nw = sqrtf(tww + 1e-10f), nc = sqrtf(tcc + 1e-10f);
  const float l1 = twc / (nw * nc), l2 = tcc / (nc * nc);
  al = g1 / (nw * nc);
  be = -(g1 * l1) / (nw * nw);
  ga = (2.f * g2 * (1.f - l2) - g1 * l1) / (nc * nc);
}

// pass 1 after cosine_partials_tma_kernel: the slots added in the order of cosine_finalize_kernel, then the coefficients
__global__ void __launch_bounds__(256) cosine_coef_finalize_kernel(const __grid_constant__ CosParams P, int grid_main,
                                                                   const float* __restrict__ gl, float* __restrict__ coef) {
  const long long total = (long long)P.N * P.HW;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int n = (int)(i / P.HW), p = (int)(i - (long long)n * P.HW);
    const int first = cos_owner((long long)n * P.chunks, P.items, grid_main);
    const int last = cos_owner((long long)n * P.chunks + P.chunks - 1, P.items, grid_main);
    float tww = 0.f, tcc = 0.f, twc = 0.f;
    for (int j = 0; j <= last - first; ++j) {
      const float* src = P.part + ((size_t)n * P.slots + j) * 3 * P.HW;
      tww += src[p];
      tcc += src[P.HW + p];
      twc += src[2 * P.HW + p];
    }
    float al, be, ga;
    cosine_coefficients(tww, tcc, twc, gl[((size_t)n * 2) * P.HW + p], gl[((size_t)n * 2 + 1) * P.HW + p], al, be, ga);
    coef[((size_t)n * 3 + 0) * P.HW + p] = al;
    coef[((size_t)n * 3 + 1) * P.HW + p] = be;
    coef[((size_t)n * 3 + 2) * P.HW + p] = ga;
  }
}

// pass 1 where the forward runs cosine_logits_nchw_kernel: the same block shape and sums
__global__ void __launch_bounds__(32 * kCosGroups) cosine_coef_nchw_kernel(const float* __restrict__ ew, const float* __restrict__ ec,
                                                                           const float* __restrict__ gl, float* __restrict__ coef,
                                                                           int E, int HW) {
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
    float al, be, ga;
    cosine_coefficients(tww, tcc, twc, gl[((size_t)n * 2) * HW + p], gl[((size_t)n * 2 + 1) * HW + p], al, be, ga);
    coef[((size_t)n * 3 + 0) * HW + p] = al;
    coef[((size_t)n * 3 + 1) * HW + p] = be;
    coef[((size_t)n * 3 + 2) * HW + p] = ga;
  }
}

struct CosBwdParams {
  CosParams C;                   // the pre-pass plan: items = (frame, pair of channels), stages, pair / stage bytes
  const float* coef;             // [N][3][HW] alpha, beta, gamma
  const unsigned char* bypass;   // (N,) or NULL: frames whose gradients are 0 (write) or left alone (add)
  float* gw;                     // d/d(emb_warp) or NULL
  float* gc;                     // d/d(emb_cur) or NULL
  int add_w, add_c;
};

__device__ __forceinline__ void cos_grad(float al, float be, float ga, float a, float b, float& vw, float& vc) {
  vw = fmaf(al, b, be * a);
  vc = fmaf(al, a, ga * b);
}

// Pass 2, all-TMA: one producer lane bulk-copies the (a, b) channel-plane pairs of an item into a stage ring, 15
// consumer warps overwrite them in place with (grad_warp, grad_cur) and the producer bulk-stores the stage
// (cp.reduce.async.bulk .add.f32 for req = add).  Measured at 64 x 2048 x 38x63 on a B200 (1000 W): 1.21 ms in place +
// bulk store, 1.31 ms with the consumers storing to global memory themselves (st.global.cs / read-add-write).
template <int PPT>
__global__ void __launch_bounds__(kTmaThreads, 1) cosine_backward_tma_kernel(const __grid_constant__ CosBwdParams B) {
  const CosParams& P = B.C;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  uint64_t* full = reinterpret_cast<uint64_t*>(smem_raw);
  uint64_t* done = full + kMaxStages;
  unsigned char* ring = smem_raw + kTmaHeaderBytes;
  const int tid = threadIdx.x, warp = tid >> 5;
  const long long i0 = P.items * (long long)blockIdx.x / gridDim.x, i1 = P.items * (long long)(blockIdx.x + 1) / gridDim.x;
  if (tid == 0) {
    for (int s = 0; s < P.stages; ++s) {
      mbar_init(&full[s], 1);
      mbar_init(&done[s], kTmaConsumerWarps);
    }
    fence_barrier_init();
  }
  __syncthreads();

  if (warp == kTmaConsumerWarps) {
    if ((tid & 31) == 0) {
      auto load = [&](long long i, int s) {
        unsigned char* st = ring + (size_t)s * P.stage_bytes;
        const size_t off = (size_t)i * 2 * P.HW;                   // planes are contiguous over (n, e)
        mbar_expect_tx(&full[s], 2u * P.pair_bytes);
        bulk_g2s(st, P.ew + off, P.pair_bytes, &full[s]);
        bulk_g2s(st + P.stage_bytes / 2, P.ec + off, P.pair_bytes, &full[s]);
      };
      long long next = i0;
      for (int s = 0; s < P.stages && next < i1; ++s) load(next++, s);
      int s = 0;
      unsigned ph = 0;
      for (long long i = i0; i < i1; ++i) {
        mbar_wait(&done[s], ph);                                   // the consumers are done with stage s
        unsigned char* st = ring + (size_t)s * P.stage_bytes;
        const size_t off = (size_t)i * 2 * P.HW;
        const bool byp = B.bypass != nullptr && B.bypass[i / P.chunks] != 0;
        if (B.gw && !(byp && B.add_w)) {
          if (B.add_w) bulk_reduce_add_s2g(B.gw + off, st, P.pair_bytes);
          else bulk_s2g(B.gw + off, st, P.pair_bytes);
        }
        if (B.gc && !(byp && B.add_c)) {
          if (B.add_c) bulk_reduce_add_s2g(B.gc + off, st + P.stage_bytes / 2, P.pair_bytes);
          else bulk_s2g(B.gc + off, st + P.stage_bytes / 2, P.pair_bytes);
        }
        bulk_commit();
        if (next < i1) {
          bulk_wait_read_all();                                    // the stores have read the stage
          load(next++, s);
        }
        if (++s == P.stages) {
          s = 0;
          ph ^= 1u;
        }
      }
      bulk_wait_all();
    }
    return;
  }

  float al[PPT], be[PPT], ga[PPT];
  bool byp = false;
  int s = 0, cur_n = -1;
  unsigned ph = 0;
  for (long long i = i0; i < i1; ++i) {
    const int n = (int)(i / P.chunks);
    if (n != cur_n) {                                              // a frame change: this frame's coefficients
      cur_n = n;
      byp = B.bypass != nullptr && B.bypass[n] != 0;
#pragma unroll
      for (int j = 0; j < PPT; ++j) {
        const int p = tid + j * kTmaConsumers;
        const bool ok = p < P.HW;
        al[j] = ok ? B.coef[((size_t)n * 3 + 0) * P.HW + p] : 0.f;
        be[j] = ok ? B.coef[((size_t)n * 3 + 1) * P.HW + p] : 0.f;
        ga[j] = ok ? B.coef[((size_t)n * 3 + 2) * P.HW + p] : 0.f;
      }
    }
    mbar_wait(&full[s], ph);
    float* a_s = reinterpret_cast<float*>(ring + (size_t)s * P.stage_bytes);
    float* b_s = reinterpret_cast<float*>(ring + (size_t)s * P.stage_bytes + P.stage_bytes / 2);
#pragma unroll
    for (int k = 0; k < 2; ++k) {
#pragma unroll
      for (int j = 0; j < PPT; ++j) {
        const int p = tid + j * kTmaConsumers;
        if (p < P.HW) {
          float vw, vc;
          cos_grad(al[j], be[j], ga[j], a_s[k * P.HW + p], b_s[k * P.HW + p], vw, vc);
          if (byp) vw = vc = 0.f;
          a_s[k * P.HW + p] = vw;
          b_s[k * P.HW + p] = vc;
        }
      }
    }
    fence_proxy_async_smem();                                      // generic-proxy writes -> the bulk store
    __syncwarp();
    if ((tid & 31) == 0) mbar_arrive(&done[s]);
    if (++s == P.stages) {
      s = 0;
      ph ^= 1u;
    }
  }
}

// Pass 2 for the shapes the TMA plan rejects (planes above 4,320 pixels, odd E or HW, misaligned pointers):
// block = 256 pixels x 32 channels of one frame
constexpr int kCosBwdThreads = 256, kCosBwdCH = 32;
__global__ void __launch_bounds__(kCosBwdThreads) cosine_backward_nchw_kernel(const __grid_constant__ CosBwdParams B) {
  const int n = blockIdx.z, HW = B.C.HW, E = B.C.E;
  const int p = blockIdx.x * kCosBwdThreads + threadIdx.x;
  if (p >= HW) return;
  const bool byp = B.bypass != nullptr && B.bypass[n] != 0;
  float* gw = (byp && B.add_w) ? nullptr : B.gw;
  float* gc = (byp && B.add_c) ? nullptr : B.gc;
  const float al = B.coef[((size_t)n * 3 + 0) * HW + p], be = B.coef[((size_t)n * 3 + 1) * HW + p],
              ga = B.coef[((size_t)n * 3 + 2) * HW + p];
  const int e1 = min(E, (int)(blockIdx.y + 1) * kCosBwdCH);
#pragma unroll 4
  for (int e = blockIdx.y * kCosBwdCH; e < e1; ++e) {
    const size_t i = ((size_t)n * E + e) * HW + p;
    float vw, vc;
    cos_grad(al, be, ga, ldg_stream(B.C.ew + i), ldg_stream(B.C.ec + i), vw, vc);
    if (byp) vw = vc = 0.f;
    if (gw) gw[i] = B.add_w ? gw[i] + vw : vw;
    if (gc) gc[i] = B.add_c ? gc[i] + vc : vc;
  }
}

static size_t up256(size_t v) { return (v + 255) & ~(size_t)255; }

size_t cosine_backward_workspace_bytes(int N, int E, int HW) {
  return up256((size_t)N * 3 * HW * sizeof(float)) + up256(cosine_tma_workspace_bytes(N, E, HW));
}

// kernel: 0 auto, 1 the plain kernel, 2 the all-TMA kernel or cudaErrorNotSupported (checked before anything is
// enqueued).  tma_sums = false pins pass 1 to the LDG form
// (what the forward ran when its all-TMA pre-pass was switched off).
cudaError_t launch_cosine_backward_nchw(const float* ew, const float* ec, const float* gl, const unsigned char* bypass, float* gw,
                                       float* gc, int add_w, int add_c, int N, int E, int HW, void* workspace,
                                       size_t workspace_bytes, bool tma_sums, int kernel, cudaStream_t st) {
  if (workspace_bytes < cosine_backward_workspace_bytes(N, E, HW) || (reinterpret_cast<uintptr_t>(workspace) % 16))
    return cudaErrorInvalidValue;
  CosBwdParams B{};
  int grid = 0, ppt = 0;
  size_t smem = 0;
  const bool tma_ok = plan_cosine_tma(ew, ec, N, E, HW, B.C, &grid, &smem, &ppt) &&
                      (reinterpret_cast<uintptr_t>(gw) % 16) == 0 && (reinterpret_cast<uintptr_t>(gc) % 16) == 0;
  if (kernel == 2 && !tma_ok) return cudaErrorNotSupported;
  B.C.ew = ew; B.C.ec = ec; B.C.N = N; B.C.E = E; B.C.HW = HW;
  float* coef = static_cast<float*>(workspace);
  char* part = static_cast<char*>(workspace) + up256((size_t)N * 3 * HW * sizeof(float));
  B.coef = coef; B.bypass = bypass; B.gw = gw; B.gc = gc; B.add_w = add_w; B.add_c = add_c;

  // pass 1: the forward's sums, then (alpha, beta, gamma)
  CosParams S;
  int sgrid = 0, sppt = 0;
  size_t ssmem = 0;
  cudaError_t e;
  if (tma_sums && plan_cosine_tma(ew, ec, N, E, HW, S, &sgrid, &ssmem, &sppt)) {
    S.part = reinterpret_cast<float*>(part);
    if (sppt == 5) {
      if ((e = cudaFuncSetAttribute(cosine_partials_tma_kernel<5>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ssmem)) != cudaSuccess) return e;
      cosine_partials_tma_kernel<5><<<sgrid, kTmaThreads, ssmem, st>>>(S);
    } else {
      if ((e = cudaFuncSetAttribute(cosine_partials_tma_kernel<9>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ssmem)) != cudaSuccess) return e;
      cosine_partials_tma_kernel<9><<<sgrid, kTmaThreads, ssmem, st>>>(S);
    }
    if ((e = cudaPeekAtLastError()) != cudaSuccess) return e;
    const long long total = (long long)N * HW;
    long long fg = (total + 255) / 256;
    if (fg > 148 * 8) fg = 148 * 8;
    cosine_coef_finalize_kernel<<<(unsigned)fg, 256, 0, st>>>(S, sgrid, gl, coef);
  } else {
    dim3 g1((HW + 31) / 32, N);
    if (g1.y > 65535) return cudaErrorInvalidValue;
    cosine_coef_nchw_kernel<<<g1, 32 * kCosGroups, 0, st>>>(ew, ec, gl, coef, E, HW);
  }
  if ((e = cudaPeekAtLastError()) != cudaSuccess) return e;

  // pass 2: the gradients
  if (kernel != 1 && tma_ok) {
    auto go = [&](auto kfn) -> cudaError_t {
      cudaError_t r = cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
      if (r != cudaSuccess) return r;
      kfn<<<grid, kTmaThreads, smem, st>>>(B);
      return cudaPeekAtLastError();
    };
    return ppt == 5 ? go(cosine_backward_tma_kernel<5>) : go(cosine_backward_tma_kernel<9>);
  }
  dim3 g2((HW + kCosBwdThreads - 1) / kCosBwdThreads, (E + kCosBwdCH - 1) / kCosBwdCH, N);
  if (g2.y > 65535 || g2.z > 65535) return cudaErrorInvalidValue;
  cosine_backward_nchw_kernel<<<g2, kCosBwdThreads, 0, st>>>(B);
  return cudaPeekAtLastError();
}

}  // namespace lsfa
