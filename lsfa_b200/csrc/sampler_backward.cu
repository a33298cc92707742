// Backward of GridGenerator(warp) + BilinearSampler (SURVEY.md 8f rank 4): what
// get_train_symbol needs from SYM:305-307 (flow_grid / flow_warping_feat: gradients to the old key
// feature AND to FlowNet's flow) and SYM:319-321 (motion_grid / motion_warping_feat: gradient to
// conv_feat only - the motion vector is data).  MXNet: src/operator/bilinear_sampler.cc
// BilinearSamplerBackward, grid_generator-inl.h Backward (kWarp).
//
// MXNet's GPU kernel scatters with one atomicAdd per tap per element.  On B200 that is the wrong
// shape for NCHW: 4 atomics per 4-byte element, and shared-memory float atomics are CAS loops
// (ATOMS.CAST.SPIN, ~2 cycles/lane).  bwd_nchw_gather_kernel turns the scatter into a GATHER:
//
//   pre-pass (bwd_lists_kernel, once per frame, channel independent): invert the sampling map - for
//     every INPUT pixel q the list of (output pixel p, tap weight) that touch it, sorted by (p, tap)
//     (= the order MXNet's sequential CPU loop adds them), stored slot-major (ELL, L slots, 6 B per
//     entry); entries beyond L go, in order, to an overflow list (served by a small ordered fix-up kernel);
//     plus a 16-byte record per OUTPUT pixel for the grid gradient (top-left weights, 4 tap offsets).
//   main kernel (same all-TMA warp-specialised pipeline as agg_nchw_tma_kernel): per (frame, K
//     channels) the producer lane TMA-loads the data planes and the out_grad planes into a stage;
//     phase A: each consumer thread accumulates d/d(grid) of its output pixels in registers
//     (4 smem taps + 1 out_grad per element); phase B: each thread owns input pixels and sums its
//     list against the out_grad planes in smem, writing grad_data IN PLACE over the data planes;
//     the producer TMA-stores them (cp.reduce.async.bulk ... add.f32 for req = kAddTo).
//   HBM: out_grad once, data once (only when d/d(grid) is wanted), grad_data once: 3F (or 2F).
//   grad_data is deterministic (fixed summation order) for any sampling map: lists longer than L are rebuilt / split in
//   (p, tap) order by the pre-pass and their tails are added by one thread per channel (bwd_overflow_kernel).
#include <cstdlib>
#include <cstring>

#include "aggregate_nchw_tma.cuh"

namespace lsfa {

struct BwdParams {
  int N, C, H, W, HW;        // out_grad / grid dims
  int Hk, Wk, HWk;           // data / grad_data plane dims
  const float* data;
  const float* coords;       // grid (N,2,H,W) normalised, or flow (feature cells) when coords_is_flow
  int coords_is_flow;
  const float* og;
  float* gdata;              // may be NULL
  float* ggrid;              // may be NULL; holds d/d(flow) when coords_is_flow
  int add_data;
  float half_w, half_h, wk_m1, hk_m1;
  // plane-resident gather kernel
  int K, chunks, L, stages;
  unsigned stage_bytes, off_og, pair_k_bytes, pair_o_bytes;
  unsigned short* ell_off;   // [N][L][HWk]  (p << 2) | tap
  float* ell_w;              // [N][L][HWk]
  unsigned char* ell_cnt;    // [N][HWk]     min(count, L)
  uint4* rec;                // [N][HW]      {wx, wy, off00|off01<<16, off10|off11<<16}, bit 0 of an offset = tap inside
  unsigned* ovf_count;       // [0] entries, [1] groups
  uint4* ovf;                // {n, q, p, weight bits}: the entries of one input pixel are contiguous and in (p, tap) order
  unsigned ovf_cap;
  uint4* ovf_groups;         // {n, q, first entry, entries}: one per input pixel whose list is longer than L
  unsigned ovf_gcap;
  int LP;                    // lists pre-pass: slots per input pixel in shared memory (>= L): what is sorted without a rescan
  unsigned* sched;
  long long pool_base;       // items [0,pool_base) split statically, the rest claimed from sched[0]
};

struct BwdTaps {
  float wx, wy;
  float w[4];                // tap weights 00,01,10,11 (0 for taps outside the plane)
  int q[4];                  // clamped element index inside a data plane
  bool ok[4];                // tap inside the plane
};

__device__ __forceinline__ BwdTaps bwd_taps(const BwdParams& P, int n, int p) {
  const float* c = P.coords + (size_t)n * 2 * P.HW;
  float gx = __ldg(c + p), gy = __ldg(c + P.HW + p);
  if (P.coords_is_flow) {
    const int y = p / P.W, x = p - y * P.W;
    gx = exact_grid(gx, (float)x, P.half_w);
    gy = exact_grid(gy, (float)y, P.half_h);
  }
  const float xr = exact_denorm(gx, P.wk_m1), yr = exact_denorm(gy, P.hk_m1);
  const int x0 = exact_floor_index(xr), y0 = exact_floor_index(yr);
  BwdTaps t;
  t.wx = exact_tl_weight(xr, x0);
  t.wy = exact_tl_weight(yr, y0);
  const double owx = 1.0 - (double)t.wx, owy = 1.0 - (double)t.wy;
  const bool xl = (x0 >= 0) && (x0 <= P.Wk - 1), xh = (x0 + 1 >= 0) && (x0 + 1 <= P.Wk - 1);
  const bool yl = (y0 >= 0) && (y0 <= P.Hk - 1), yh = (y0 + 1 >= 0) && (y0 + 1 <= P.Hk - 1);
  t.ok[0] = xl && yl; t.ok[1] = xh && yl; t.ok[2] = xl && yh; t.ok[3] = xh && yh;
  t.w[0] = t.ok[0] ? (float)((double)t.wy * (double)t.wx) : 0.0f;
  t.w[1] = t.ok[1] ? (float)((double)t.wy * owx) : 0.0f;
  t.w[2] = t.ok[2] ? (float)(owy * (double)t.wx) : 0.0f;
  t.w[3] = t.ok[3] ? (float)(owy * owx) : 0.0f;
  const int xa = min(max(x0, 0), P.Wk - 1), xb = min(max(x0 + 1, 0), P.Wk - 1);
  const int ya = min(max(y0, 0), P.Hk - 1), yb = min(max(y0 + 1, 0), P.Hk - 1);
  t.q[0] = ya * P.Wk + xa; t.q[1] = ya * P.Wk + xb; t.q[2] = yb * P.Wk + xa; t.q[3] = yb * P.Wk + xb;
  return t;
}

// d(out)/d(grid) scale of BilinearSamplerBackward (`gw * (i_w - 1) / 2`), followed by GridGenerator's
// backward (`grad / ((W-1)/2)`) when the coordinates were given as a flow
__device__ __forceinline__ float grid_grad_scale(float g, float dim_m1, bool is_flow, float half) {
  float v = __fdiv_rn(__fmul_rn(g, dim_m1), 2.0f);
  if (is_flow) v = __fdiv_rn(v, half);
  return v;
}

// ---------------------------------------------------------------------------------------
// Generic scatter kernel (any shape): one thread per output pixel and group of channels,
// atomics into grad_data / grad_grid - MXNet's own GPU formulation; fallback and ablation.
// ---------------------------------------------------------------------------------------
constexpr int kBwdGenericThreads = 256;
constexpr int kBwdGenericCG = 32;

__global__ void __launch_bounds__(kBwdGenericThreads) bwd_generic_kernel(const __grid_constant__ BwdParams P) {
  const int n = blockIdx.z;
  const int p = blockIdx.x * kBwdGenericThreads + threadIdx.x;
  if (p >= P.HW) return;
  const int c0 = blockIdx.y * kBwdGenericCG, c1 = min(P.C, c0 + kBwdGenericCG);
  const BwdTaps t = bwd_taps(P, n, p);
  float gxa = 0.f, gya = 0.f;
  for (int c = c0; c < c1; ++c) {
    const float og = __ldg(P.og + ((size_t)n * P.C + c) * P.HW + p);
    const size_t pl = ((size_t)n * P.C + c) * P.HWk;
    if (P.gdata) {
#pragma unroll
      for (int k = 0; k < 4; ++k)
        if (t.ok[k] && t.w[k] != 0.0f) atomicAdd(P.gdata + pl + t.q[k], t.w[k] * og);
    }
    if (P.ggrid) {
      const float v00 = t.ok[0] ? __ldg(P.data + pl + t.q[0]) : 0.f, v01 = t.ok[1] ? __ldg(P.data + pl + t.q[1]) : 0.f;
      const float v10 = t.ok[2] ? __ldg(P.data + pl + t.q[2]) : 0.f, v11 = t.ok[3] ? __ldg(P.data + pl + t.q[3]) : 0.f;
      const float d = v00 - v01 - v10 + v11;
      gya -= og * (v01 - v11 + d * t.wx);
      gxa -= og * (v10 - v11 + d * t.wy);
    }
  }
  if (P.ggrid) {
    atomicAdd(P.ggrid + ((size_t)n * 2 + 0) * P.HW + p, grid_grad_scale(gxa, P.wk_m1, P.coords_is_flow, P.half_w));
    atomicAdd(P.ggrid + ((size_t)n * 2 + 1) * P.HW + p, grid_grad_scale(gya, P.hk_m1, P.coords_is_flow, P.half_h));
  }
}

// ---------------------------------------------------------------------------------------
// Pre-pass: inverse sampling lists + grid-gradient records, one CTA per frame.
// ---------------------------------------------------------------------------------------
constexpr int kBwdListThreads = 512;

__global__ void __launch_bounds__(kBwdListThreads) bwd_lists_kernel(const __grid_constant__ BwdParams P) {
  extern __shared__ __align__(16) unsigned char lsm[];
  int* cnt = reinterpret_cast<int*>(lsm);                                   // [HWk]
  float* w_s = reinterpret_cast<float*>(lsm + (size_t)((P.HWk + 3) / 4 * 4) * 4);   // [LP][HWk]
  unsigned short* o_s = reinterpret_cast<unsigned short*>(w_s + (size_t)P.LP * P.HWk);   // [LP][HWk]
  const int n = blockIdx.x, tid = threadIdx.x;
  const bool lists = P.gdata != nullptr;
  if (lists)
    for (int q = tid; q < P.HWk; q += kBwdListThreads) cnt[q] = 0;
  __syncthreads();
  for (int p = tid; p < P.HW; p += kBwdListThreads) {
    const BwdTaps t = bwd_taps(P, n, p);
    if (P.ggrid) {
      unsigned o[4];
#pragma unroll
      for (int k = 0; k < 4; ++k) o[k] = ((unsigned)t.q[k] << 2) | (t.ok[k] ? 1u : 0u);
      P.rec[(size_t)n * P.HW + p] = make_uint4(__float_as_uint(t.wx), __float_as_uint(t.wy), o[0] | (o[1] << 16), o[2] | (o[3] << 16));
    }
    if (lists) {
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        if (!t.ok[k] || t.w[k] == 0.0f) continue;        // a zero weight adds nothing
        const int slot = atomicAdd(&cnt[t.q[k]], 1);
        if (slot < P.LP) {                               // LP >= L slots here; lists beyond LP are rebuilt in order below
          w_s[(size_t)slot * P.HWk + t.q[k]] = t.w[k];
          o_s[(size_t)slot * P.HWk + t.q[k]] = (unsigned short)(((unsigned)p << 2) | (unsigned)k);
        }
      }
    }
  }
  if (!lists) return;
  __syncthreads();
  // Determinism for ANY sampling map.  A list of up to LP entries is complete in shared memory: sorted by (p, tap) below,
  // its first L entries go to the slots and the rest, in order, to one contiguous group of the overflow list.  For a list
  // longer than LP, WHICH entries won a slot depends on the order of the atomics: one warp rebuilds it in (p, tap) order
  // by scanning the taps of every output pixel (rare: LP is 12-15 at 38x63).  The fix-up kernel adds a group's entries
  // in that order from one thread per channel.
  {
    const int lane = tid & 31, warp = tid >> 5;
    for (int q = warp; q < P.HWk; q += kBwdListThreads / 32) {
      const int total = cnt[q];
      if (total <= P.LP) continue;
      const unsigned n_over = (unsigned)(total - P.L);
      unsigned start = 0u;
      if (lane == 0) {
        start = atomicAdd(P.ovf_count, n_over);
        const unsigned g = atomicAdd(P.ovf_count + 1, 1u);
        if (g < P.ovf_gcap) P.ovf_groups[g] = make_uint4((unsigned)n, (unsigned)q, start, n_over);
      }
      start = __shfl_sync(0xffffffffu, start, 0);
      int pos = 0;
      for (int p0 = 0; p0 < P.HW; p0 += 32) {
        const int p = p0 + lane;
        bool hit[4] = {false, false, false, false};
        float hw[4] = {0.f, 0.f, 0.f, 0.f};
        if (p < P.HW) {
          const BwdTaps t = bwd_taps(P, n, p);
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            hit[k] = t.ok[k] && t.w[k] != 0.0f && t.q[k] == q;
            hw[k] = t.w[k];
          }
        }
        const int nh = (int)hit[0] + (int)hit[1] + (int)hit[2] + (int)hit[3];
        int incl = nh;                                   // inclusive prefix over the lanes = over p
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
          const int v = __shfl_up_sync(0xffffffffu, incl, o);
          if (lane >= o) incl += v;
        }
        int j = pos + incl - nh;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          if (!hit[k]) continue;
          if (j < P.L) {
            w_s[(size_t)j * P.HWk + q] = hw[k];
            o_s[(size_t)j * P.HWk + q] = (unsigned short)(((unsigned)p << 2) | (unsigned)k);
          } else {
            const unsigned e = start + (unsigned)(j - P.L);
            if (e < P.ovf_cap) P.ovf[e] = make_uint4((unsigned)n, (unsigned)q, (unsigned)p, __float_as_uint(hw[k]));
          }
          ++j;
        }
        pos += __shfl_sync(0xffffffffu, incl, 31);
      }
    }
  }
  __syncthreads();
  for (int q = tid; q < P.HWk; q += kBwdListThreads) {
    const int held = min(cnt[q], P.LP);                   // entries of this list in shared memory
    const int c = min(cnt[q], P.L);
    // sort the column by (p, tap): MXNet's sequential loop adds in exactly this order (rebuilt columns already are)
    for (int i = 1; i < held && cnt[q] <= P.LP; ++i) {
      const unsigned short ko = o_s[(size_t)i * P.HWk + q];
      const float kw = w_s[(size_t)i * P.HWk + q];
      int j = i - 1;
      while (j >= 0 && o_s[(size_t)j * P.HWk + q] > ko) {
        o_s[(size_t)(j + 1) * P.HWk + q] = o_s[(size_t)j * P.HWk + q];
        w_s[(size_t)(j + 1) * P.HWk + q] = w_s[(size_t)j * P.HWk + q];
        --j;
      }
      o_s[(size_t)(j + 1) * P.HWk + q] = ko;
      w_s[(size_t)(j + 1) * P.HWk + q] = kw;
    }
    if (cnt[q] > P.L && cnt[q] <= P.LP) {                // the tail of a complete list: one ordered overflow group
      const unsigned n_over = (unsigned)(cnt[q] - P.L);
      const unsigned start = atomicAdd(P.ovf_count, n_over);
      const unsigned g = atomicAdd(P.ovf_count + 1, 1u);
      if (g < P.ovf_gcap) P.ovf_groups[g] = make_uint4((unsigned)n, (unsigned)q, start, n_over);
      for (int i = P.L; i < cnt[q]; ++i) {
        const unsigned e = start + (unsigned)(i - P.L);
        const unsigned key = o_s[(size_t)i * P.HWk + q];
        if (e < P.ovf_cap) P.ovf[e] = make_uint4((unsigned)n, (unsigned)q, key >> 2, __float_as_uint(w_s[(size_t)i * P.HWk + q]));
      }
    }
    P.ell_cnt[(size_t)n * P.HWk + q] = (unsigned char)c;
    for (int s = 0; s < P.L; ++s) {   // unused slots: weight 0, offset 0 (never read: loops stop at the count)
      const bool used = s < c;
      P.ell_w[((size_t)n * P.L + s) * P.HWk + q] = used ? w_s[(size_t)s * P.HWk + q] : 0.0f;
      P.ell_off[((size_t)n * P.L + s) * P.HWk + q] = used ? o_s[(size_t)s * P.HWk + q] : (unsigned short)0;
    }
  }
}

// list entries that did not fit the L slots: one thread per (input pixel group, channel) adds the group's entries in
// their (p, tap) order and then adds the sum to grad_data[n,c,q] - the only thread that touches that element after the
// gather kernel: deterministic
__global__ void __launch_bounds__(256) bwd_overflow_kernel(const __grid_constant__ BwdParams P) {
  const unsigned groups = min(P.ovf_count[1], P.ovf_gcap);
  const long long total = (long long)groups * P.C;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const unsigned g = (unsigned)(i % groups);
    const int c = (int)(i / groups);
    const uint4 gr = P.ovf_groups[g];
    const size_t fc = (size_t)gr.x * P.C + c;
    const unsigned end = min(gr.z + gr.w, P.ovf_cap);
    float acc = 0.f;
    for (unsigned e = gr.z; e < end; ++e) {
      const uint4 v = P.ovf[e];
      acc = fmaf(__uint_as_float(v.w), __ldg(P.og + fc * P.HW + v.z), acc);
    }
    P.gdata[fc * P.HWk + gr.y] += acc;
  }
}

__device__ __forceinline__ void consumer_bar() { asm volatile("bar.sync 1, %0;" ::"n"(kTmaConsumers) : "memory"); }

// ---------------------------------------------------------------------------------------
// Main kernel: plane-resident gather.
// ---------------------------------------------------------------------------------------
// predicated shared-memory load: no access when on == false (the result is then 0), no branch
__device__ __forceinline__ float lds_f32_if(unsigned addr, bool on) {
  float v;
  asm volatile("{\n .reg .pred q;\n setp.ne.u32 q, %2, 0;\n mov.f32 %0, 0f00000000;\n @q ld.shared.f32 %0, [%1];\n}"
               : "=f"(v)
               : "r"(addr), "r"((unsigned)on));
  return v;
}

template <int K, int PPT, int LR>
__global__ void __launch_bounds__(kTmaThreads, 1) bwd_nchw_gather_kernel(const __grid_constant__ BwdParams P) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  uint64_t* full = reinterpret_cast<uint64_t*>(smem_raw);
  uint64_t* done = full + kMaxStages;
  volatile int2* desc = reinterpret_cast<volatile int2*>(smem_raw + 128);
  unsigned char* ring = smem_raw + kTmaHeaderBytes;
  float* ellw_s = reinterpret_cast<float*>(ring + (size_t)P.stages * P.stage_bytes);                   // [L-LR][HWk]
  unsigned short* ello_s = reinterpret_cast<unsigned short*>(ellw_s + (size_t)(P.L - LR) * P.HWk);     // [L-LR][HWk]
  const int tid = threadIdx.x, warp = tid >> 5;
  const bool has_data = P.gdata != nullptr, has_grid = P.ggrid != nullptr;

  if (tid == 0) {
    for (int s = 0; s < P.stages; ++s) {
      mbar_init(&full[s], 1);
      mbar_init(&done[s], kTmaConsumerWarps);
    }
    fence_barrier_init();
  }
  __syncthreads();

  if (warp == kTmaConsumerWarps) {
    // =========================== producer warp (one elected lane) ===========================
    if ((tid & 31) == 0) {
      // work source, as in agg_nchw_tma_kernel: a static contiguous share of the (frame, chunk) items per CTA
      // (few frame changes: a change reloads the lists), then a pool claimed kTmaClaim at a time from one counter
      unsigned* sched = P.sched;
      const long long items = (long long)P.N * P.chunks;
      const long long pool_base = sched ? P.pool_base : items;
      long long lin = pool_base * (long long)blockIdx.x / gridDim.x;
      long long lin_end = pool_base * (long long)(blockIdx.x + 1) / gridDim.x;
      bool pool_open = sched != nullptr && pool_base < items;
      auto next_item = [&](int& n, int& chunk) -> bool {
        while (true) {
          if (lin < lin_end) {
            n = (int)(lin / P.chunks);
            chunk = (int)(lin - (long long)n * P.chunks);
            ++lin;
            return true;
          }
          if (!pool_open) return false;
          const long long got = pool_base + (long long)atomicAdd(sched, (unsigned)kTmaClaim);
          if (got >= items) {
            pool_open = false;
            return false;
          }
          lin = got;
          lin_end = min(got + (long long)kTmaClaim, items);
        }
      };
      auto issue_loads = [&](int s, int n, int chunk) {
        unsigned char* st = ring + (size_t)s * P.stage_bytes;
        desc[s].x = n;
        desc[s].y = chunk;
        mbar_expect_tx(&full[s], P.pair_o_bytes + (has_grid ? P.pair_k_bytes : 0u));
        const size_t pl = (size_t)n * P.C + (size_t)chunk * K;
        if (has_grid) bulk_g2s(st, P.data + pl * P.HWk, P.pair_k_bytes, &full[s]);
        bulk_g2s(st + P.off_og, P.og + pl * P.HW, P.pair_o_bytes, &full[s]);
      };
      auto issue_store = [&](int s) {
        if (!has_data) return;
        const size_t pl = (size_t)desc[s].x * P.C + (size_t)desc[s].y * K;
        unsigned char* st = ring + (size_t)s * P.stage_bytes;
        if (P.add_data) bulk_reduce_add_s2g(P.gdata + pl * P.HWk, st, P.pair_k_bytes);
        else bulk_s2g(P.gdata + pl * P.HWk, st, P.pair_k_bytes);
        bulk_commit();
      };
      auto issue_stop = [&](int s) {
        desc[s].x = -1;
        desc[s].y = 0;
        mbar_arrive(&full[s]);
      };
      int n, chunk, live = 0;
      bool stopped = false;
      for (int s = 0; s < P.stages; ++s) {
        if (next_item(n, chunk)) {
          issue_loads(s, n, chunk);
          ++live;
        } else {
          issue_stop(s);
          stopped = true;
          break;
        }
      }
      int s = 0;
      unsigned ph = 0;
      while (live > 0) {
        mbar_wait(&done[s], ph);
        issue_store(s);
        --live;
        if (!stopped) {
          if (next_item(n, chunk)) {
            bulk_wait_read_all();
            issue_loads(s, n, chunk);
            ++live;
          } else {
            issue_stop(s);
            stopped = true;
          }
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

  // ================================= consumer warps ==========================================
  // Per-thread state, rebuilt at every frame change:
  //   output-pixel slots (phase A): top-left weights, 4 packed tap offsets, running d/d(grid) sums;
  //   input-pixel slots (phase B): the first LR list entries in REGISTERS (weight + packed 16-bit out_grad
  //   offset), entries LR..L-1 in shared memory (ELL), the list length.
  float wx[PPT], wy[PPT], gxa[PPT], gya[PPT];
  unsigned ot[PPT], ob[PPT];
  constexpr int LRP = LR > 0 ? LR : 1, LRH = LR > 0 ? (LR + 1) / 2 : 1;
  float lw[PPT][LRP];
  unsigned lo[PPT][LRH];
  int cq[PPT];
#pragma unroll
  for (int j = 0; j < PPT; ++j) {
    wx[j] = wy[j] = gxa[j] = gya[j] = 0.f;
    ot[j] = ob[j] = 0u;
    cq[j] = 0;
#pragma unroll
    for (int e = 0; e < LRP; ++e) lw[j][e] = 0.f;
#pragma unroll
    for (int e = 0; e < LRH; ++e) lo[j][e] = 0u;
  }
  const int LS = P.L - LR;            // list slots kept in shared memory (>= 0 by planning)
  int cur_n = -1, s = 0;
  unsigned ph = 0, inside = 0u;   // bit j: every tap of slot j is inside the plane for the whole warp
  const unsigned og_plane_bytes = (unsigned)P.HW * 4u;
  auto flush = [&](int n) {
#pragma unroll
    for (int j = 0; j < PPT; ++j) {
      const int p = tid + j * kTmaConsumers;
      if (p < P.HW) {
        atomicAdd(P.ggrid + ((size_t)n * 2 + 0) * P.HW + p, grid_grad_scale(gxa[j], P.wk_m1, P.coords_is_flow, P.half_w));
        atomicAdd(P.ggrid + ((size_t)n * 2 + 1) * P.HW + p, grid_grad_scale(gya[j], P.hk_m1, P.coords_is_flow, P.half_h));
      }
      gxa[j] = gya[j] = 0.f;
    }
  };
  while (true) {
    mbar_wait(&full[s], ph);
    const int n = desc[s].x;
    if (n < 0) break;
    if (n != cur_n) {
      if (cur_n >= 0 && has_grid) flush(cur_n);
      cur_n = n;
      if (has_data) {
        const float* gw = P.ell_w + (size_t)n * P.L * P.HWk;
        const unsigned short* go = P.ell_off + (size_t)n * P.L * P.HWk;
        if (LS > 0) {
          consumer_bar();        // every consumer is done with the previous frame's lists
          const int tot = LS * P.HWk, skip = LR * P.HWk;
          for (int i = tid; i < tot; i += kTmaConsumers) {
            ellw_s[i] = __ldg(gw + skip + i);
            ello_s[i] = __ldg(go + skip + i);
          }
          consumer_bar();
        }
#pragma unroll
        for (int j = 0; j < PPT; ++j) {
          const int q = tid + j * kTmaConsumers;
          const bool in = q < P.HWk;
          cq[j] = in ? (int)__ldg(P.ell_cnt + (size_t)n * P.HWk + q) : 0;
          if (LR > 0) {
#pragma unroll
            for (int e = 0; e < LRH; ++e) lo[j][e] = 0u;
#pragma unroll
            for (int e = 0; e < LR; ++e) {
              const bool use = in && e < P.L;
              lw[j][e] = use ? __ldg(gw + (size_t)e * P.HWk + q) : 0.f;
              const unsigned o = use ? ((unsigned)__ldg(go + (size_t)e * P.HWk + q) & 0xfffcu) : 0u;
              lo[j][e >> 1] |= o << ((e & 1) * 16);
            }
          }
        }
      }
      if (has_grid) {
#pragma unroll
        for (int j = 0; j < PPT; ++j) {
          const int p = tid + j * kTmaConsumers;
          uint4 r = make_uint4(0u, 0u, 0u, 0u);
          if (p < P.HW) r = __ldg(P.rec + (size_t)n * P.HW + p);
          wx[j] = __uint_as_float(r.x);
          wy[j] = __uint_as_float(r.y);
          ot[j] = r.z;
          ob[j] = r.w;
          const bool all4 = (r.z & r.w & 0x10001u) == 0x10001u || p >= P.HW;
          inside = (inside & ~(1u << j)) | (__all_sync(0xffffffffu, all4) ? (1u << j) : 0u);
        }
      }
    }
    unsigned char* st = ring + (size_t)s * P.stage_bytes;
    const unsigned char* og_s = st + P.off_og;
    if (has_grid) {
      // ---- phase A: d/d(grid) of this thread's output pixels (reads the data planes) ----
#pragma unroll
      for (int k = 0; k < K; ++k) {
        const unsigned char* plane = st + (size_t)k * P.HWk * 4;
        const float* ogk = reinterpret_cast<const float*>(og_s + (size_t)k * P.HW * 4);
#pragma unroll
        for (int j = 0; j < PPT; ++j) {
          const int p = tid + j * kTmaConsumers;
          if (p < P.HW) {
            const float og = ogk[p];
            float v00 = *reinterpret_cast<const float*>(plane + (ot[j] & 0xfffcu));
            float v01 = *reinterpret_cast<const float*>(plane + ((ot[j] >> 16) & 0xfffcu));
            float v10 = *reinterpret_cast<const float*>(plane + (ob[j] & 0xfffcu));
            float v11 = *reinterpret_cast<const float*>(plane + ((ob[j] >> 16) & 0xfffcu));
            if (!((inside >> j) & 1u)) {   // uniform per warp: some lane of this slot has a tap outside the plane
              v00 = (ot[j] & 1u) ? v00 : 0.f;
              v01 = (ot[j] & 0x10000u) ? v01 : 0.f;
              v10 = (ob[j] & 1u) ? v10 : 0.f;
              v11 = (ob[j] & 0x10000u) ? v11 : 0.f;
            }
            const float d = v00 - v01 - v10 + v11;
            gya[j] -= og * (v01 - v11 + d * wx[j]);
            gxa[j] -= og * (v10 - v11 + d * wy[j]);
          }
        }
      }
      if (has_data) consumer_bar();   // all taps read before grad_data overwrites the data planes
    }
    if (has_data) {
      // ---- phase B: grad_data of this thread's input pixels, gathered through its list ----
      const unsigned og_a = smem_u32(og_s);
#pragma unroll
      for (int j = 0; j < PPT; ++j) {
        const int q = tid + j * kTmaConsumers;
        const int c = cq[j];
        const int m = __reduce_max_sync(0xffffffffu, c);   // warp-uniform trip count
        float acc[K];
#pragma unroll
        for (int k = 0; k < K; ++k) acc[k] = 0.f;
#pragma unroll
        for (int g = 0; g < LR; g += 3) {
          if (g < m) {   // uniform branch; three entries at a time: all shared loads first, then the FMAs
            float v[3][K];
#pragma unroll
            for (int u = 0; u < 3; ++u) {
              const int e = g + u;
              if (e < LR) {
                const unsigned off = (lo[j][e >> 1] >> ((e & 1) * 16)) & 0xffffu;
#pragma unroll
                for (int k = 0; k < K; ++k)   // lanes whose list is shorter have weight 0: predicated off, no access
                  v[u][k] = lds_f32_if(og_a + (unsigned)k * og_plane_bytes + off, lw[j][e] != 0.0f);
              }
            }
#pragma unroll
            for (int u = 0; u < 3; ++u) {
              const int e = g + u;
              if (e < LR) {
#pragma unroll
                for (int k = 0; k < K; ++k) acc[k] = fmaf(lw[j][e], v[u][k], acc[k]);
              }
            }
          }
        }
        for (int e = LR; e < m; ++e) {                     // the tail of long lists: entries in shared memory
          const int i = (e - LR) * P.HWk + q;
          const bool on = e < c;
          const unsigned off = on ? ((unsigned)ello_s[i] & 0xfffcu) : 0u;
          const float w = on ? ellw_s[i] : 0.f;
#pragma unroll
          for (int k = 0; k < K; ++k) acc[k] = fmaf(w, lds_f32_if(og_a + (unsigned)k * og_plane_bytes + off, on), acc[k]);
        }
        if (q < P.HWk) {
#pragma unroll
          for (int k = 0; k < K; ++k) reinterpret_cast<float*>(st + (size_t)k * P.HWk * 4)[q] = acc[k];
        }
      }
      fence_proxy_async_smem();
    }
    __syncwarp();
    if ((tid & 31) == 0) mbar_arrive(&done[s]);
    if (++s == P.stages) {
      s = 0;
      ph ^= 1u;
    }
  }
  if (cur_n >= 0 && has_grid) flush(cur_n);
}

// ---------------------------------------------------------------------------------------
// grid_generator backward (kWarp): gdata = grad / ((dim - 1) / 2)
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) grid_generator_warp_backward_kernel(const float* __restrict__ g, float* __restrict__ o,
                                                                           long long total, int HW, float half_w,
                                                                           float half_h, int add) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int ch = (int)((i / HW) & 1);
    float v = __fdiv_rn(__ldg(g + i), ch ? half_h : half_w);
    if (add) v += o[i];
    o[i] = v;
  }
}

// ---------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------
static size_t r16(size_t v) { return (v + 15) / 16 * 16; }
constexpr int kBwdMaxL = 8;
constexpr int kBwdRegSlots = 6;   // list entries per input pixel kept in registers by the PPT = 5 kernel

size_t bwd_workspace_bytes(int N, int HWk, int HW) {
  return r16((size_t)N * 4) + 16 + r16((size_t)N * HW * 16) + r16((size_t)N * kBwdMaxL * HWk * 2) +
         r16((size_t)N * kBwdMaxL * HWk * 4) + r16((size_t)N * HWk) + (size_t)N * HW * 4 * 16 + (size_t)N * HWk * 16;
}

static bool plan_bwd_gather(BwdParams& P, size_t* smem_main, size_t* smem_lists, int* ppt_out) {
  const size_t kSmemMax = 227 * 1024;
  const int max_pix = 9 * kTmaConsumers;
  if (P.HW > max_pix || P.HWk > max_pix) return false;
  const void* ptrs[3] = {P.data, P.og, P.gdata};
  for (const void* q : ptrs)
    if (q && (reinterpret_cast<uintptr_t>(q) % 16)) return false;
  int K = 0;
  if (P.C % 2 == 0 && (2LL * P.HWk) % 4 == 0 && (2LL * P.HW) % 4 == 0) K = 2;
  else if (P.HWk % 4 == 0 && P.HW % 4 == 0) K = 1;
  if (K == 0) return false;
  P.K = K;
  P.chunks = P.C / K;
  P.pair_k_bytes = (unsigned)((size_t)K * P.HWk * 4);
  P.pair_o_bytes = (unsigned)((size_t)K * P.HW * 4);
  P.off_og = (P.pair_k_bytes + 127u) / 128u * 128u;
  P.stage_bytes = P.off_og + (P.pair_o_bytes + 127u) / 128u * 128u;
  // PPT = 5 (planes up to 2400 pixels): the first 6 list entries live in registers, only slots 6.. need shared
  // memory; PPT = 9: every slot in shared memory
  const int ppt = (P.HW <= 5 * kTmaConsumers && P.HWk <= 5 * kTmaConsumers) ? 5 : 9;
  const int LR = ppt == 5 ? kBwdRegSlots : 0;
  const int lcand5[6] = {8, 8, 6, 6, 6, 6}, scand5[6] = {5, 4, 5, 4, 3, 2};
  const int lcand9[6] = {6, 6, 4, 4, 3, 2}, scand9[6] = {3, 2, 3, 2, 2, 2};
  const int nolist_stages[6] = {5, 4, 4, 3, 2, 2};
  const bool lists = P.gdata != nullptr;
  for (int i = 0; i < 6; ++i) {
    const int L = lists ? (ppt == 5 ? lcand5[i] : lcand9[i]) : LR;
    const int S = lists ? (ppt == 5 ? scand5[i] : scand9[i]) : nolist_stages[i];
    const size_t need = kTmaHeaderBytes + (size_t)S * P.stage_bytes + r16((size_t)(L - LR) * P.HWk * 6);
    if (need > kSmemMax) continue;
    P.L = L;
    P.stages = S;
    *smem_main = need;
    *smem_lists = (size_t)((P.HWk + 3) / 4 * 4) * 4 + r16((size_t)L * P.HWk * 6);
    *ppt_out = ppt;
    return true;
  }
  return false;
}

template <int K, int PPT>
static cudaError_t launch_gather(const BwdParams& P, size_t smem, int grid, cudaStream_t st) {
  auto kfn = bwd_nchw_gather_kernel<K, PPT, (PPT == 5 ? kBwdRegSlots : 0)>;
  cudaError_t e = cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  kfn<<<grid, kTmaThreads, smem, st>>>(P);
  return cudaPeekAtLastError();
}

static int bwd_sm_count() {
  int dev = 0, n = 148;
  if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
  return n > 0 ? n : 148;
}

// kernel: 0 auto, 1 generic scatter, 2 gather (fails with cudaErrorNotSupported if it cannot serve the args)
cudaError_t launch_sampler_backward(const float* data, const float* coords, int coords_is_flow, const float* og,
                                    float* gdata, float* ggrid, int N, int C, int Hi, int Wi, int Ho, int Wo,
                                    int add_data, int add_grid, float half_w, float half_h, void* workspace,
                                    size_t workspace_bytes, int kernel, cudaStream_t st) {
  BwdParams P;
  memset(&P, 0, sizeof(P));
  P.N = N; P.C = C; P.H = Ho; P.W = Wo; P.HW = Ho * Wo;
  P.Hk = Hi; P.Wk = Wi; P.HWk = Hi * Wi;
  P.data = data; P.coords = coords; P.coords_is_flow = coords_is_flow; P.og = og;
  P.gdata = gdata; P.ggrid = ggrid; P.add_data = add_data;
  P.half_w = half_w; P.half_h = half_h; P.wk_m1 = (float)(Wi - 1); P.hk_m1 = (float)(Hi - 1);
  const int sm_count = bwd_sm_count();
  cudaError_t e;
  size_t smem_main = 0, smem_lists = 0;
  int ppt = 5;
  const bool ws_ok = workspace && workspace_bytes >= bwd_workspace_bytes(P.N, P.HWk, P.HW) &&
                     (reinterpret_cast<uintptr_t>(workspace) % 16) == 0;
  // decide the kernel BEFORE touching any output: an unsupported request must leave the caller's buffers alone
  const bool gather = kernel != 1 && ws_ok && plan_bwd_gather(P, &smem_main, &smem_lists, &ppt);
  if (kernel == 2 && !gather) return cudaErrorNotSupported;
  if (P.ggrid && !add_grid) {
    e = cudaMemsetAsync(P.ggrid, 0, (size_t)P.N * 2 * P.HW * sizeof(float), st);
    if (e != cudaSuccess) return e;
  }
  if (gather) {
    char* ws = static_cast<char*>(workspace);
    P.sched = reinterpret_cast<unsigned*>(ws);
    ws += r16((size_t)P.N * 4);
    P.ovf_count = reinterpret_cast<unsigned*>(ws);
    ws += 16;
    P.rec = reinterpret_cast<uint4*>(ws);
    ws += r16((size_t)P.N * P.HW * 16);
    P.ell_off = reinterpret_cast<unsigned short*>(ws);
    ws += r16((size_t)P.N * kBwdMaxL * P.HWk * 2);
    P.ell_w = reinterpret_cast<float*>(ws);
    ws += r16((size_t)P.N * kBwdMaxL * P.HWk * 4);
    P.ell_cnt = reinterpret_cast<unsigned char*>(ws);
    ws += r16((size_t)P.N * P.HWk);
    P.ovf = reinterpret_cast<uint4*>(ws);
    P.ovf_cap = (unsigned)((size_t)P.N * P.HW * 4);
    ws += (size_t)P.N * P.HW * 4 * 16;
    P.ovf_groups = reinterpret_cast<uint4*>(ws);
    P.ovf_gcap = (unsigned)((size_t)P.N * P.HWk);
    {   // pre-pass slots: as many as fit the shared memory (complete lists need no rescan), at least L
      const size_t cnt_bytes = (size_t)((P.HWk + 3) / 4 * 4) * 4;
      long long lp = ((long long)227 * 1024 - (long long)cnt_bytes - 16) / ((long long)P.HWk * 6);
      if (lp > 16) lp = 16;
      if (lp < P.L) lp = P.L;
      P.LP = (int)lp;
      smem_lists = cnt_bytes + r16((size_t)P.LP * P.HWk * 6);
    }
    e = cudaMemsetAsync(workspace, 0, r16((size_t)P.N * 4) + 16, st);   // claim counters + overflow count
    if (e != cudaSuccess) return e;
    e = cudaFuncSetAttribute(bwd_lists_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_lists);
    if (e != cudaSuccess) return e;
    bwd_lists_kernel<<<P.N, kBwdListThreads, smem_lists, st>>>(P);
    e = cudaPeekAtLastError();
    if (e != cudaSuccess) return e;
    long long grid = sm_count;
    const long long items = (long long)P.N * P.chunks;
    if (grid > items) grid = items;
    {
      int pct = kTmaPoolPercent;
      if (const char* e = knob("LSFA_TMA_POOL_PCT")) pct = atoi(e);
      pct = pct < 0 ? 0 : (pct > 100 ? 100 : pct);
      P.pool_base = items - items * pct / 100;
      P.pool_base -= P.pool_base % kTmaClaim;
    }
    if (P.K == 2 && ppt == 5) e = launch_gather<2, 5>(P, smem_main, (int)grid, st);
    else if (P.K == 2) e = launch_gather<2, 9>(P, smem_main, (int)grid, st);
    else if (ppt == 5) e = launch_gather<1, 5>(P, smem_main, (int)grid, st);
    else e = launch_gather<1, 9>(P, smem_main, (int)grid, st);
    if (e != cudaSuccess) return e;
    if (P.gdata) {
      bwd_overflow_kernel<<<2 * sm_count, 256, 0, st>>>(P);
      e = cudaPeekAtLastError();
    }
    return e;
  }
  if (P.gdata && !P.add_data) {
    e = cudaMemsetAsync(P.gdata, 0, (size_t)P.N * P.C * P.HWk * sizeof(float), st);
    if (e != cudaSuccess) return e;
  }
  dim3 grid((P.HW + kBwdGenericThreads - 1) / kBwdGenericThreads, (P.C + kBwdGenericCG - 1) / kBwdGenericCG, P.N);
  if (grid.y > 65535 || grid.z > 65535) return cudaErrorInvalidValue;
  bwd_generic_kernel<<<grid, kBwdGenericThreads, 0, st>>>(P);
  return cudaPeekAtLastError();
}

// how many kernels the call above enqueues (memsets not counted)
int sampler_backward_num_launches(int N, int C, int Hi, int Wi, int Ho, int Wo, bool want_data, bool ws_ok, int kernel) {
  BwdParams P;
  memset(&P, 0, sizeof(P));
  P.N = N; P.C = C; P.HW = Ho * Wo; P.HWk = Hi * Wi;
  P.gdata = want_data ? reinterpret_cast<float*>(16) : nullptr;
  size_t a = 0, b = 0;
  int ppt = 0;
  if (kernel != 1 && ws_ok && plan_bwd_gather(P, &a, &b, &ppt)) return want_data ? 3 : 2;
  return 1;
}

cudaError_t launch_grid_generator_backward(const float* g, float* o, int N, int H, int W, float half_w, float half_h,
                                           int add, cudaStream_t st) {
  const long long total = (long long)N * 2 * H * W;
  long long grid = (total + 255) / 256;
  if (grid > 148 * 8) grid = 148 * 8;
  grid_generator_warp_backward_kernel<<<(unsigned)grid, 256, 0, st>>>(g, o, total, H * W, half_w, half_h, add);
  return cudaPeekAtLastError();
}

}  // namespace lsfa
