// agg_nchw_tma_kernel - the all-TMA, warp-specialised form of the plane-resident gather.
//
// Same operator chain as agg_nchw_plane_kernel (SYM:571-576, 308/470/680, 236, 104-108,
// 144-147, 315; choose_feat.py:23-31) but NO thread ever touches global memory for the
// feature streams: a dedicated producer warp moves every byte with bulk async copies
//     HBM --cp.async.bulk (TMA, mbarrier complete_tx)--> SMEM stage {key planes, scale, cur}
//     SMEM stage {out, written in place over cur} --cp.async.bulk (TMA store, bulk_group)--> HBM
// and 16 consumer warps do shared-memory-only work (4 gather taps + 2 streaming loads + 1
// store per element).  Why it beats the LDG/STG form: NCHW planes of 38x63 floats start at
// 8-byte phases inside 32-byte DRAM sectors, so every warp-wide 128-byte global access
// straddles a sector that its neighbour warp touches again; with evict-first streams the
// second touch often misses L2 (+14% DRAM reads measured).  TMA reads each 19 KB chunk once.
//
// Pipeline (S stages, S >= 2):  full[s]  : producer -> consumers   (TMA bytes landed)
//                               done[s]  : consumers -> producer   (stage computed, out in smem)
//   producer: wait done[c] -> TMA-store stage c -> wait_group.read -> TMA-load the next item into it
// Work: a static contiguous share per CTA followed by a dynamically claimed pool (one counter in a
// caller-supplied scratch) so that SMs that finish early take the tail; each stage carries its
// (frame, chunk) descriptor in smem.
#pragma once
#include <cooperative_groups.h>

#include "aggregate_nchw_plane.cuh"

namespace lsfa {

constexpr int kTmaConsumers = 480;   // 15 warps: 480 x 5 = 2400 slots for 38x63 = 2394 pixels
constexpr int kTmaConsumerWarps = kTmaConsumers / 32;
constexpr int kTmaThreads = kTmaConsumers + 32;   // + one producer warp

__device__ __forceinline__ void bulk_s2g(void* dst_gmem, const void* src_smem, uint32_t bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst_gmem),
               "r"(smem_u32(src_smem)), "r"(bytes)
               : "memory");
}
// element-wise out += smem (req = kAddTo): one contributor per element, so the result is deterministic
__device__ __forceinline__ void bulk_reduce_add_s2g(void* dst_gmem, const void* src_smem, uint32_t bytes) {
  asm volatile("cp.reduce.async.bulk.global.shared::cta.bulk_group.add.f32 [%0], [%1], %2;" ::"l"(dst_gmem),
               "r"(smem_u32(src_smem)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_read_all() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

constexpr int kTmaHeaderBytes = 256;   // 16 mbarriers + one item descriptor per stage
constexpr int kTmaClaim = 4;           // items per dynamic claim (4 x ~1.8 us of work)
constexpr int kTmaPoolPercent = 10;    // share of the items left to the dynamic pool (see the producer)
constexpr int kCoopMaxVirtualFrames = 8;   // up to this many (frame, pixel part) pairs: the one-launch cooperative form

// The 15 consumer warps of both all-TMA kernels (single CTA and 2-CTA cluster): shared-memory-only
// work on the stages the producer warp fills.  fixed_part < 0: the stage descriptor carries a virtual
// frame (frame * parts + part); fixed_part >= 0 (cluster kernel): it carries the frame, and this CTA
// always works on pixel part `fixed_part`.
template <int K, int PPT, int VAR, bool DIRECT>
__device__ __forceinline__ void tma_consumer_loop(const AggParams& P, uint64_t* full, uint64_t* done, volatile int2* desc,
                                                  unsigned char* ring, float* res_s, float4* rnet_s, const int tid,
                                                  const int fixed_part) {
  constexpr bool has_scale = VAR == kVarScale || VAR == kVarScaleCur;
  constexpr bool has_cur = VAR == kVarScaleCur || VAR == kVarResCur;
  constexpr bool has_res = VAR == kVarResCur;
  const bool has_bypass = P.bypass != nullptr;
  // ================================= consumer warps ==========================================
  float w00[PPT], w01[PPT], w10[PPT], w11[PPT], wc[PPT], ww[PPT];
  // tap byte offsets inside a key plane: (i00 | i01 << 16), (i10 | i11 << 16).  Warp-only variant (P.canon): the record is
  // canonical (canonical_taps: the 2x2 block at o_top's low half, rows row_bytes apart), which saves the unpacking -
  // measured +2.6 % there; the same form costs the HBM-bound headline variant 2.2 % (denser LDS bursts), so it keeps
  // the packed offsets.
  unsigned o_top[PPT], o_bot[PPT];
  constexpr bool canon = DIRECT;       // = the warp-only variant of agg_nchw_tma_kernel; its launcher sets P.canon for the pre-pass
  const unsigned row_bytes = (unsigned)P.Wk * 4u;
  unsigned valid = 0;
  int cur_vf = -1, n = 0;
  bool byp = false;
  int s = 0;
  unsigned ph = 0;
  const unsigned plane_bytes = (unsigned)P.HWk * 4u;
  const unsigned io_plane_bytes = (unsigned)(P.parts == 1 ? P.HW : P.part_pix) * 4u;
  (void)ww;
  constexpr int JG = PPT > 5 ? 3 : PPT;   // pixel slots handled together (bounds the live registers)
  // pooled residual of this thread's pixels (a10): in registers for up to 5 slots - three shared-memory reads per
  // element less on the variant that is shared-memory-bandwidth bound; larger parts keep it in smem
  constexpr bool RES_REG = has_res && PPT <= 5;
  constexpr int RRN = RES_REG ? PPT : 1;
  float rr0[RRN], rr1[RRN], rr2[RRN];
#pragma unroll
  for (int j = 0; j < RRN; ++j) rr0[j] = rr1[j] = rr2[j] = 0.f;

  if (has_res) {   // the 1x1 conv's weights (SYM:66) sit in smem: per-item global loads would stall every item
    for (int c = tid; c < P.C; c += kTmaConsumers)
      rnet_s[c] = make_float4(__ldg(P.rnet_w + (size_t)c * 3), __ldg(P.rnet_w + (size_t)c * 3 + 1),
                              __ldg(P.rnet_w + (size_t)c * 3 + 2), __ldg(P.rnet_b + c));
    asm volatile("bar.sync 1, %0;" ::"n"(kTmaConsumers) : "memory");   // consumers only (the producer warp is elsewhere)
  }

  while (true) {
    mbar_wait(&full[s], ph);
    const int vf = desc[s].x;
    if (vf < 0) break;
    const int chunk = desc[s].y;
    if (vf != cur_vf) {  // new frame (or pixel part): rebuild this thread's sampling records
      cur_vf = vf;
      int part;
      if (fixed_part >= 0) {
        n = vf;
        part = fixed_part;
      } else {
        n = vf / P.parts;
        part = vf - n * P.parts;
      }
      const int pix0 = part * P.part_pix;
      const int pend = min(P.HW, pix0 + P.part_pix);
      byp = has_bypass && (__ldg(P.bypass + n) != 0);
      valid = 0;
      if (P.records != nullptr) {
        // records come from the pre-pass (agg_records_kernel) or, cooperative form, from this launch's own consumers
        // before the grid barrier: two 16-byte loads per pixel slot, from L2 (never the non-coherent path)
        uint4 ra[PPT], rb[PPT];
#pragma unroll
        for (int j = 0; j < PPT; ++j) {
          const int p = pix0 + tid + j * kTmaConsumers;
          ra[j] = rb[j] = make_uint4(0u, 0u, 0u, 0u);
          if (p < pend) {
            valid |= 1u << j;
            if (!byp) {
              const uint4* rp = P.records + 2 * ((size_t)n * P.HW + p);
              ra[j] = __ldcg(rp);
              rb[j] = __ldcg(rp + 1);
            }
          }
        }
#pragma unroll
        for (int j = 0; j < PPT; ++j) {
          w00[j] = __uint_as_float(ra[j].x); w01[j] = __uint_as_float(ra[j].y);
          w10[j] = __uint_as_float(ra[j].z); w11[j] = __uint_as_float(ra[j].w);
          wc[j] = __uint_as_float(rb[j].x); ww[j] = __uint_as_float(rb[j].y);
          o_top[j] = rb[j].z; o_bot[j] = rb[j].w;
          if (has_res) {
            const int p = pix0 + tid + j * kTmaConsumers;
            if (p < pend && !byp) {
              if (RES_REG) {
                rr0[j % RRN] = __ldg(P.res + ((size_t)n * 3 + 0) * P.HW + p);
                rr1[j % RRN] = __ldg(P.res + ((size_t)n * 3 + 1) * P.HW + p);
                rr2[j % RRN] = __ldg(P.res + ((size_t)n * 3 + 2) * P.HW + p);
              } else {
#pragma unroll
                for (int k = 0; k < 3; ++k)
                  res_s[k * (PPT * kTmaConsumers) + (p - pix0)] = __ldg(P.res + ((size_t)n * 3 + k) * P.HW + p);
              }
            }
          }
        }
      } else {
      // the old records are dead from here on: clearing them first frees their registers for the
      // load batch below (otherwise ptxas spills the batch and every spill store waits on its load)
#pragma unroll
      for (int j = 0; j < PPT; ++j) {
        w00[j] = w01[j] = w10[j] = w11[j] = wc[j] = ww[j] = 0.0f;
        o_top[j] = o_bot[j] = 0u;      // slot outside the part: taps read offset 0, store is predicated off
      }
      // phase A0: L2 prefetch of everything the records need, all pixel slots back to back
      if (!byp) {
#pragma unroll
        for (int j = 0; j < PPT; ++j) {
          const int p = pix0 + tid + j * kTmaConsumers;
          if (p < pend) prefetch_pixel_loads(P, n, p / P.W, p % P.W);
        }
      }
      // phase A: the loads proper, a few pixel slots at a time (they now hit in L2)
      constexpr int RG = PPT >= 3 ? 3 : PPT;              // slots per load batch (register budget)
#pragma unroll
      for (int j0 = 0; j0 < PPT; j0 += RG) {
        PixelLoads ld[RG];
#pragma unroll
        for (int g = 0; g < RG; ++g) {
          const int j = j0 + g;
          const int p = pix0 + tid + j * kTmaConsumers;
          if (j < PPT && p < pend && !byp) ld[g] = issue_pixel_loads(P, n, p / P.W, p % P.W);
        }
        // phase B: the arithmetic (float64 pooling, exact fp32 grid round trip, softmax, fold)
#pragma unroll
        for (int g = 0; g < RG; ++g) {
          const int j = j0 + g;
          if (j >= PPT) continue;
          const int p = pix0 + tid + j * kTmaConsumers;
          if (p < pend) {
            valid |= 1u << j;
            if (!byp) {
              PixelRec t = finish_pixel(P, ld[g], n, p / P.W, p % P.W);
              if (canon) canonical_taps(t, P.Hk, P.Wk);
              w00[j] = t.w00; w01[j] = t.w01; w10[j] = t.w10; w11[j] = t.w11;
              wc[j] = t.wc; ww[j] = t.ww;
              o_top[j] = (unsigned)(t.i00 * 4) | ((unsigned)(t.i01 * 4) << 16);
              o_bot[j] = (unsigned)(t.i10 * 4) | ((unsigned)(t.i11 * 4) << 16);
              if (has_res) {
                if (RES_REG) {
                  rr0[j % RRN] = __ldg(P.res + ((size_t)n * 3 + 0) * P.HW + p);
                  rr1[j % RRN] = __ldg(P.res + ((size_t)n * 3 + 1) * P.HW + p);
                  rr2[j % RRN] = __ldg(P.res + ((size_t)n * 3 + 2) * P.HW + p);
                } else {
#pragma unroll
                  for (int k = 0; k < 3; ++k)
                    res_s[k * (PPT * kTmaConsumers) + (p - pix0)] = __ldg(P.res + ((size_t)n * 3 + k) * P.HW + p);
                }
              }
            }
          }
        }
      }
      }  // in-kernel record build
    }

    if (!byp) {   // bypass frames: cur already sits in the io buffer, it is stored back as is
      unsigned char* stage_s = ring + (size_t)s * P.stage_bytes;
      const int c0 = chunk * K;
      // variants without a current feature may skip the shared-memory staging of the output (one STS and one
      // copy-engine read per element less on the variants that are shared-memory-bandwidth bound)
      constexpr bool direct = DIRECT;
      float* out_g = nullptr;
      if (direct) {
        const int part_d = fixed_part >= 0 ? fixed_part : cur_vf - n * P.parts;
        out_g = static_cast<float*>(P.out) + ((size_t)n * P.C + c0) * P.HW + (size_t)part_d * P.part_pix + tid;
      }
#pragma unroll
      for (int k = 0; k < K; ++k) {
        float rw0 = 0.f, rw1 = 0.f, rw2 = 0.f, rb = 0.f;
        if (has_res) {
          const float4 rw = rnet_s[c0 + k];   // broadcast read
          rw0 = rw.x; rw1 = rw.y; rw2 = rw.z; rb = rw.w;
        }
        const unsigned char* plane_s = stage_s + (size_t)k * plane_bytes;
        const float* sc_s = reinterpret_cast<const float*>(stage_s + P.off_scale + (size_t)k * io_plane_bytes) + tid;
        float* io_s = reinterpret_cast<float*>(stage_s + P.off_io + (size_t)k * io_plane_bytes) + tid;
#pragma unroll
        for (int j0 = 0; j0 < PPT; j0 += JG) {
          float v00[JG], v01[JG], v10[JG], v11[JG], sc[JG], cu[JG];
#pragma unroll
          for (int g = 0; g < JG; ++g) {   // all shared-memory reads of the group first ...
            const int j = j0 + g;
            if (j < PPT) {
              if (canon) {
                const unsigned char* top = plane_s + (o_top[j] & 0xffffu);   // the 2x2 block: two adds, four loads at +0 / +4
                const unsigned char* bot = top + row_bytes;
                v00[g] = *reinterpret_cast<const float*>(top);
                v01[g] = *reinterpret_cast<const float*>(top + 4);
                v10[g] = *reinterpret_cast<const float*>(bot);
                v11[g] = *reinterpret_cast<const float*>(bot + 4);
              } else {
                v00[g] = *reinterpret_cast<const float*>(plane_s + (o_top[j] & 0xffffu));
                v01[g] = *reinterpret_cast<const float*>(plane_s + (o_top[j] >> 16));
                v10[g] = *reinterpret_cast<const float*>(plane_s + (o_bot[j] & 0xffffu));
                v11[g] = *reinterpret_cast<const float*>(plane_s + (o_bot[j] >> 16));
              }
              const bool ok = (valid >> j) & 1u;   // slots past the plane are neither read nor written (a read there would
                                                   // land in the next plane, which its owner rewrites in place)
              sc[g] = (has_scale && ok) ? sc_s[j * kTmaConsumers] : 1.0f;
              cu[g] = (has_cur && ok) ? io_s[j * kTmaConsumers] : 0.0f;
            }
          }
#pragma unroll
          for (int g = 0; g < JG; ++g) {   // ... then the arithmetic and the in-place stores
            const int j = j0 + g;
            if (j < PPT) {
              float v = w00[j] * v00[g];
              v = fmaf(w01[j], v01[g], v);
              v = fmaf(w10[j], v10[g], v);
              v = fmaf(w11[j], v11[g], v);
              if (has_scale) v *= sc[g];
              if (has_res) {
                const int q = tid + j * kTmaConsumers;
                if (RES_REG)
                  v = fmaf(ww[j], rnet_term(rw0, rw1, rw2, rb, rr0[j % RRN], rr1[j % RRN], rr2[j % RRN]), v);
                else
                  v = fmaf(ww[j], rnet_term(rw0, rw1, rw2, rb, res_s[q], res_s[PPT * kTmaConsumers + q],
                                            res_s[2 * PPT * kTmaConsumers + q]), v);
              }
              const float o = has_cur ? fmaf(wc[j], cu[g], v) : v;
              if ((valid >> j) & 1u) {
                if (direct) stg_stream(out_g + (size_t)k * P.HW + j * kTmaConsumers, o);
                else io_s[j * kTmaConsumers] = o;
              }
            }
          }
        }
      }
      if (!direct) fence_proxy_async_smem();   // generic-proxy writes -> visible to the TMA store
    }
    __syncwarp();
    if ((tid & 31) == 0) mbar_arrive(&done[s]);
    if (++s == P.stages) {
      s = 0;
      ph ^= 1u;
    }
  }
}

template <int K, int PPT, int VAR>
__global__ void __launch_bounds__(kTmaThreads, 1)
agg_nchw_tma_kernel(const __grid_constant__ AggParams P) {
  static_assert(VAR != kVarRuntime, "the TMA kernel is only built for the compile-time variants");
  constexpr bool has_scale = VAR == kVarScale || VAR == kVarScaleCur;
  constexpr bool has_cur = VAR == kVarScaleCur || VAR == kVarResCur;
  constexpr bool has_res = VAR == kVarResCur;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  uint64_t* full = reinterpret_cast<uint64_t*>(smem_raw);
  uint64_t* done = full + kMaxStages;
  volatile int2* desc = reinterpret_cast<volatile int2*>(smem_raw + 128);   // (frame, chunk) of each stage; frame < 0 = stop
  unsigned char* ring = smem_raw + kTmaHeaderBytes;
  float* res_s = reinterpret_cast<float*>(ring + (size_t)P.stages * P.stage_bytes);  // [3][PPT*480]
  float4* rnet_s = reinterpret_cast<float4*>(res_s + (PPT <= 5 ? 0 : 3 * PPT * kTmaConsumers));       // [C] (w0,w1,w2,b), res variant only

  const int tid = threadIdx.x;
  const int warp = tid >> 5;
  const bool has_bypass = P.bypass != nullptr;

  uint64_t* rec_issued = reinterpret_cast<uint64_t*>(smem_raw + 192);   // cooperative form: see the producer's first loads
  if (tid == 0) {
    for (int s = 0; s < P.stages; ++s) {
      mbar_init(&full[s], 1);
      mbar_init(&done[s], kTmaConsumerWarps);
    }
    mbar_init(rec_issued, kTmaConsumerWarps);
    fence_barrier_init();
  }
  __syncthreads();

  if (warp == kTmaConsumerWarps) {
    // =========================== producer warp (one elected lane) ===========================
    if ((tid & 31) != 0) {
      if (P.coop) cooperative_groups::this_grid().sync();     // every thread of the grid takes part in the barrier
      return;
    }
    {
      // ---- work source: a static contiguous share per CTA, then a shared pool claimed dynamically ----
      // Linear item index = virtual frame * chunks + chunk; a "virtual frame" is (frame, pixel part): planes
      // larger than PPT*480 pixels are cut into parts, each with its own sampling records and slice of the
      // scale/cur/out streams.  Items [0, pool_base) are split evenly and contiguously over the CTAs (no
      // atomics, a CTA stays on one frame for ~hundreds of items, so its per-frame records are rebuilt once or
      // twice); items [pool_base, items) are claimed kTmaClaim at a time from ONE counter, so SMs that finish
      // early (unequal GPCs, bypass frames, row-trimmed parts) take the tail.  pool_base == items: purely
      // static (no scratch given); pool_base == 0: purely dynamic.
      unsigned* sched = P.sched;
      const long long pool_base = sched ? P.pool_base : P.items;
      long long lin = pool_base * (long long)blockIdx.x / gridDim.x;
      long long lin_end = pool_base * (long long)(blockIdx.x + 1) / gridDim.x;
      bool pool_open = sched != nullptr && pool_base < P.items;
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
          if (got >= P.items) {
            pool_open = false;
            return false;
          }
          lin = got;
          lin_end = min(got + (long long)kTmaClaim, P.items);
        }
      };
      int range_vf = -1;
      uint32_t range_b0 = 0u, range_b1 = 0u;
      auto issue_loads = [&](int s, int vf, int chunk) {
        const int n = vf / P.parts, part = vf - n * P.parts;
        const bool byp = has_bypass && __ldg(P.bypass + n) != 0;
        unsigned char* st = ring + (size_t)s * P.stage_bytes;
        const int pix0 = part * P.part_pix;
        const uint32_t len_bytes = (uint32_t)(min(P.part_pix, P.HW - pix0)) * 4u;   // one plane's slice
        // parts == 1: the K planes of a stream are one contiguous run; otherwise one copy per plane
        const uint32_t io_tx = P.parts == 1 ? P.io_bytes : (uint32_t)K * len_bytes;
        const size_t e0 = ((size_t)n * P.C + (size_t)chunk * K) * P.HW + pix0;
        // key bytes of one plane this part needs: whole plane, or (row-trimmed) the 16-byte-rounded span of the
        // rows its taps read - copied to the SAME smem offsets, so the tap offsets in the records stay valid
        uint32_t kb0 = 0u, kb1 = (uint32_t)P.HWk * 4u;
        const bool trimmed = P.rowrange != nullptr;
        if (trimmed && !byp) {
          if (vf != range_vf) {
            range_vf = vf;
            const unsigned hi = __ldcg(P.rowrange + 2 * vf), lo_inv = __ldcg(P.rowrange + 2 * vf + 1);
            range_b0 = hi ? (((uint32_t)(P.Hk - (int)lo_inv) * (uint32_t)P.Wk * 4u) & ~15u) : 0u;
            range_b1 = hi ? min((uint32_t)P.HWk * 4u, (hi * (uint32_t)P.Wk * 4u + 15u) & ~15u) : 0u;
          }
          kb0 = range_b0;
          kb1 = range_b1;
        }
        const uint32_t key_tx = trimmed ? (uint32_t)K * (kb1 - kb0) : P.key_bytes;
        uint32_t bytes = has_cur ? io_tx : 0u;
        if (!byp) bytes += key_tx + (has_scale ? io_tx : 0u);
        desc[s].x = vf;
        desc[s].y = chunk;
        mbar_expect_tx(&full[s], bytes);              // release: the descriptor is visible with the data
        if (!byp) {
          const int kn = key_slot(P, n);
          const float* ksrc = static_cast<const float*>(P.key) + ((size_t)kn * P.C + (size_t)chunk * K) * P.HWk;
          if (!trimmed) {
            bulk_g2s(st, ksrc, P.key_bytes, &full[s]);
          } else if (kb1 > kb0) {
#pragma unroll
            for (int k = 0; k < K; ++k)
              bulk_g2s(st + (size_t)k * P.HWk * 4 + kb0, reinterpret_cast<const unsigned char*>(ksrc + (size_t)k * P.HWk) + kb0,
                       kb1 - kb0, &full[s]);
          }
        }
        if (P.parts == 1) {
          if (!byp && has_scale) bulk_g2s(st + P.off_scale, static_cast<const float*>(P.scale) + e0, P.io_bytes, &full[s]);
          if (has_cur) bulk_g2s(st + P.off_io, static_cast<const float*>(P.cur) + e0, P.io_bytes, &full[s]);
        } else {
#pragma unroll
          for (int k = 0; k < K; ++k) {
            const size_t ek = e0 + (size_t)k * P.HW;
            const uint32_t dk = (uint32_t)k * (uint32_t)P.part_pix * 4u;
            if (!byp && has_scale) bulk_g2s(st + P.off_scale + dk, static_cast<const float*>(P.scale) + ek, len_bytes, &full[s]);
            if (has_cur) bulk_g2s(st + P.off_io + dk, static_cast<const float*>(P.cur) + ek, len_bytes, &full[s]);
          }
        }
      };
      auto issue_store = [&](int s) {
        const int vf = desc[s].x, chunk = desc[s].y;
        const int n = vf / P.parts, part = vf - n * P.parts;
        const int pix0 = part * P.part_pix;
        unsigned char* st = ring + (size_t)s * P.stage_bytes;
        float* dst = static_cast<float*>(P.out) + ((size_t)n * P.C + (size_t)chunk * K) * P.HW + pix0;
        if (P.parts == 1) {
          bulk_s2g(dst, st + P.off_io, P.io_bytes);
        } else {
          const uint32_t len_bytes = (uint32_t)(min(P.part_pix, P.HW - pix0)) * 4u;
#pragma unroll
          for (int k = 0; k < K; ++k)
            bulk_s2g(dst + (size_t)k * P.HW, st + P.off_io + (uint32_t)k * (uint32_t)P.part_pix * 4u, len_bytes);
        }
        bulk_commit();
      };
      auto issue_stop = [&](int s) {
        desc[s].x = -1;
        desc[s].y = 0;
        mbar_arrive(&full[s]);
      };

      int n, chunk;
      int live = 0;                                    // stages holding a real item
      bool stopped = false;
      // cooperative form: the handful of loads the record math starts from (a few KB for the whole grid) are the head of the
      // launch's critical path (loads -> index math -> grid barrier -> first item); issued after this CTA's share of the
      // ~25 MB stage prefetch they queue behind it and land 1-2 us late, so the prefetch waits until they are out
      if (P.coop) mbar_wait(rec_issued, 0u);
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
      // cooperative form: the first stages are already in flight while the consumers of the whole grid build the records
      if (P.coop) cooperative_groups::this_grid().sync();
      int s = 0;
      unsigned ph = 0;
      constexpr bool direct = VAR == kVarWarpOnly;           // the consumers wrote the output themselves
      while (live > 0) {
        mbar_wait(&done[s], ph);                       // consumers finished this stage; out is in smem
        if (!direct) issue_store(s);
        --live;
        if (!stopped) {
          if (next_item(n, chunk)) {
            if (!direct) bulk_wait_read_all();         // the store has drained the stage: safe to refill
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
      bulk_wait_all();                                 // every store is complete before the CTA exits
    }
    return;
  }

  if (P.coop) {
    // one-launch form (small batches: the reference's batch-1 mode): the index math of the whole batch - at most a pixel
    // or two per consumer thread of the grid - is done here instead of in a pre-pass kernel, then a grid-wide barrier
    // pixels are dealt out by warp, round robin over the CTAs of the grid (one frame = 75 warps: one warp in each of 75 SMs
    // instead of 15 warps in each of 5: the FP64 / division work of the index math does not queue)
    uint4* rec = const_cast<uint4*>(P.records);
    const long long total = (long long)P.N * P.HW;
    const long long step = (long long)gridDim.x * kTmaConsumerWarps * 32;
    bool told = false;
    for (long long i = ((long long)warp * gridDim.x + blockIdx.x) * 32 + (tid & 31);; i += step) {
      const bool live = i < total;
      int n = 0, p = 0;
      if (live) {
        n = (int)(i / P.HW);
        p = (int)(i - (long long)n * P.HW);
      }
      const bool work = live && !(has_bypass && __ldg(P.bypass + n) != 0);
      const int y = p / P.W, x = p - y * P.W;
      PixelLoads ld;
      if (work) ld = issue_pixel_loads(P, n, y, x);
      if (!told) {                                   // this warp's first loads are out (or it has none)
        told = true;
        __syncwarp();
        if ((tid & 31) == 0) mbar_arrive(rec_issued);
      }
      if (!__any_sync(0xffffffffu, live)) break;
      if (work) {
        PixelRec t = finish_pixel(P, ld, n, y, x);
        if (P.canon) canonical_taps(t, P.Hk, P.Wk);
        uint4 a, b;
        pack_record(t, a, b);
        __stcg(rec + 2 * i, a);
        __stcg(rec + 2 * i + 1, b);
      }
    }
    __threadfence();
    cooperative_groups::this_grid().sync();
  }
  tma_consumer_loop<K, PPT, VAR, VAR == kVarWarpOnly>(P, full, done, desc, ring, res_s, rnet_s, tid, -1);
}

template <int VAR>
cudaError_t launch_tma_variant(const AggParams& P, size_t smem, int grid, cudaStream_t st);

#define LSFA_TMA_FOREACH_KP(X) X(1, 1) X(1, 3) X(1, 5) X(1, 9) X(2, 1) X(2, 3) X(2, 5) X(2, 9)

// the opt-in to 227 KB of dynamic shared memory is a per-function, per-device attribute: set it the first time a device
// sees the instantiation, not on every launch (idempotent: a race between two host threads sets it twice)
#define LSFA_TMA_LAUNCH(VAR, KK, PP)                                                              \
  if (P.K == KK && ppt == PP) {                                                                   \
    auto kfn = agg_nchw_tma_kernel<KK, PP, VAR>;                                                  \
    static bool attr_done[64];                                                                    \
    int dev_ = 0;                                                                                 \
    cudaGetDevice(&dev_);                                                                         \
    if (dev_ < 0 || dev_ >= 64 || !attr_done[dev_]) {                                             \
      cudaError_t e = cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024); \
      if (e != cudaSuccess) return e;                                                             \
      if (dev_ >= 0 && dev_ < 64) attr_done[dev_] = true;                                         \
    }                                                                                             \
    cudaLaunchConfig_t cfg = {};                                                                  \
    cfg.gridDim = dim3((unsigned)grid);                                                           \
    cfg.blockDim = dim3(kTmaThreads);                                                             \
    cfg.dynamicSmemBytes = smem;                                                                  \
    cfg.stream = st;                                                                              \
    cudaLaunchAttribute attr[1];                                                                  \
    attr[0].id = cudaLaunchAttributeCooperative;                                                  \
    attr[0].val.cooperative = 1;                                                                  \
    cfg.attrs = attr;                                                                             \
    cfg.numAttrs = P.coop ? 1 : 0;                                                                \
    return cudaLaunchKernelEx(&cfg, kfn, P);                                                      \
  }

}  // namespace lsfa
