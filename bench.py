#!/usr/bin/env python
"""Benchmark of the non-key-frame propagation + aggregation path (BASELINE.json metric).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
  torchrun --nproc-per-node N ... bench.py --gpus N ...      (one rank per GPU, no collective
                                                              on the data path: streams shard)

One "step" = one pass of the hot path over one batch of synthetic frames:
  workload (BASELINE.json configs[1]): 64 non-key frames per GPU, C=1024, 38x63 features, fp32
  NCHW, raw 600x1000 int32 motion vectors pooled in-kernel, warp x scale map, softmax-logit
  aggregation with the current-frame feature (SURVEY.md 8d variant V2).
`value`  : whole-job frames/s with every input resident in HBM (CUDA events, max over ranks).
`e2e`    : same metric through lsfa_b200.host.HostAggregator: pinned HOST buffers in, pinned
           host buffer out, H2D/D2H inside the timed region.
`roofline`: algorithmic bytes of the fused kernel / its measured launch time vs the measured
           HBM copy bandwidth (MEASURED_PEAKS.json).
`cpu_baseline`: the reference's CPU path (C port of the MXNet CPU operators, oracle/) timed on
           this box's host cores on a bounded sample.
`--impl reference` times that CPU path alone and prints the same line with "impl":"reference".
`--dump-outputs DIR` (rank 0): after the timed steps, what each timed path returned in its last step -
           value.npy (the device output), e2e.npy and e2e_gop.npy (the host output of the two e2e rows) - as
           float32, each a fixed seeded sample of DUMP_SAMPLE values when the output is larger.  The inputs are
           seeded, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import statistics
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "non-key frames/s (warp+aggregate) @1024x38x63; achieved HBM GB/s vs peak"
UNIT = "frames/s"
C, H, W = 1024, 38, 63
MV_H, MV_W = 600, 1000
FRAMES_PER_GPU = 64
FALLBACK_HBM_GBS = 6650.0          # /opt/skills/guides/B200_PROFILING.md, used only if MEASURED_PEAKS.json is absent


def algorithmic_bytes_v2(frames, feat_bytes=4):
    """SURVEY.md 8d, V2: 4F (key, scale, cur, out) + 32*HW (4 MV taps x 2 ch x 4 B) + 8*HW (logits)."""
    F = C * H * W * feat_bytes
    return frames * (4 * F + 32 * H * W + 8 * H * W)


DUMP_SAMPLE = 4 << 20             # values per dumped output: 3 x 16 MB stays within 64 MB


def dump_sample(t):
    """float32 numpy copy of `t` (device or host tensor), or of DUMP_SAMPLE of its values when it is larger: flat indices
    drawn with a fixed seed and sorted, so every run with the same output shape samples the same elements."""
    import numpy as np
    import torch
    if t.numel() <= DUMP_SAMPLE:
        return t.float().cpu().numpy()
    idx = np.sort(np.random.default_rng(0).integers(0, t.numel(), DUMP_SAMPLE))
    return t.reshape(-1)[torch.from_numpy(idx).to(t.device)].float().cpu().numpy()


def workload_config(frames, n_gpus):
    return {
        "workload": "BASELINE configs[1]: fused MV-warp x scale + softmax-logit aggregation, %d non-key frames "
                    "per GPU, C=1024, 38x63, fp32 NCHW, raw 600x1000 int32 MVs pooled in-kernel (V2)" % frames,
        "frames_per_gpu": frames, "channels": C, "feat_h": H, "feat_w": W, "mv_h": MV_H, "mv_w": MV_W,
        "layout": "NCHW", "sharding": "independent streams per GPU, no collective" if n_gpus > 1 else "single GPU",
        "l2_policy": "per-step working set %.2f GB >> 126 MB L2 (no flush needed)" % (algorithmic_bytes_v2(frames) / 1e9),
    }


# --------------------------------------------------------------------------------------------
# clocks during the timed region (NVML in a sampling thread; nvidia-smi as a fallback)
# --------------------------------------------------------------------------------------------
REASON_BITS = {0x1: "gpu_idle", 0x2: "applications_clocks_setting", 0x4: "sw_power_cap", 0x8: "hw_slowdown",
               0x10: "sync_boost", 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown",
               0x80: "hw_power_brake_slowdown", 0x100: "display_clock_setting"}


class ClockSampler(threading.Thread):
    def __init__(self, torch_index, period_s=0.002):
        super().__init__(daemon=True)
        self.period = period_s
        self.samples, self.reasons = [], 0
        self._stop_evt = threading.Event()
        self.ok = False
        self.max_mhz = None
        try:
            import pynvml
            import torch
            pynvml.nvmlInit()
            self.nv = pynvml
            try:
                uuid = "GPU-" + str(torch.cuda.get_device_properties(torch_index).uuid)
                self.h = pynvml.nvmlDeviceGetHandleByUUID(uuid.encode() if hasattr(uuid, "encode") else uuid)
            except Exception:
                self.h = pynvml.nvmlDeviceGetHandleByIndex(torch_index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception:
            self.ok = False

    def _reasons(self):
        for name in ("nvmlDeviceGetCurrentClocksEventReasons", "nvmlDeviceGetCurrentClocksThrottleReasons"):
            fn = getattr(self.nv, name, None)
            if fn is not None:
                try:
                    return int(fn(self.h))
                except Exception:
                    pass
        return 0

    def run(self):
        if not self.ok:
            return
        while not self._stop_evt.is_set():
            try:
                self.samples.append(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM))
                self.reasons |= self._reasons()
            except Exception:
                pass
            time.sleep(self.period)

    def stop(self):
        self._stop_evt.set()
        if self.is_alive():
            self.join(timeout=2)
        if self.ok and not self.samples:
            try:
                self.samples.append(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM))
                self.reasons |= self._reasons()
            except Exception:
                pass

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["unavailable"], "samples": 0}
        names = [n for b, n in REASON_BITS.items() if self.reasons & b and n != "gpu_idle"]
        return {"sm_mhz": float(statistics.median(self.samples)), "sm_max_mhz": self.max_mhz,
                "reasons": names, "samples": len(self.samples)}


# --------------------------------------------------------------------------------------------
# synthetic inputs (SURVEY.md 8d), generated on the host into pinned memory
# --------------------------------------------------------------------------------------------
def make_host_inputs(frames, seed, pinned=True):
    import numpy as np
    import torch
    rng = np.random.default_rng(seed)

    def pin(shape, dtype):
        t = torch.empty(shape, dtype=dtype)
        return t.pin_memory() if pinned else t

    host = {"key": pin((frames, C, H, W), torch.float32), "cur": pin((frames, C, H, W), torch.float32),
            "scale_map": pin((frames, C, H, W), torch.float32), "mv": pin((frames, MV_H, MV_W, 2), torch.int32),
            "logits": pin((frames, 2, H, W), torch.float32)}
    for k in ("key", "cur"):
        a = host[k].numpy()
        rng.standard_normal(out=a, dtype=np.float32)
        np.maximum(a, 0, out=a)                      # post-ReLU features (SYM:54)
    a = host["scale_map"].numpy()
    rng.standard_normal(out=a, dtype=np.float32)
    a *= np.float32(0.1)
    a += np.float32(1.0)
    # macroblock-constant integer MVs, half the blocks static, the rest uniform in [-32,32] px
    bh, bw = -(-MV_H // 16), -(-MV_W // 16)
    blk = rng.integers(-32, 33, size=(frames, bh, bw, 2), dtype=np.int32)
    blk[rng.random((frames, bh, bw)) < 0.5] = 0
    host["mv"].numpy()[:] = np.repeat(np.repeat(blk, 16, axis=1), 16, axis=2)[:, :MV_H, :MV_W]
    rng.standard_normal(out=host["logits"].numpy(), dtype=np.float32)
    return host


# --------------------------------------------------------------------------------------------
# the reference's CPU path (C port of the MXNet CPU operators) on a bounded sample
# --------------------------------------------------------------------------------------------
def cpu_reference_fps(sample_frames, reps, warmup, seed=0):
    """frames/s of oracle/lsfa_oracle.c::lsfa_ref_chain_nq (op-by-op graph, OpenMP over all host
    threads) on `sample_frames` frames of the same workload; returns (fps, cores, ms_per_rep)."""
    import numpy as np
    from oracle import c_port
    c_port.build()
    c_port.use_all_cores()
    host = make_host_inputs(sample_frames, seed, pinned=False)
    arr = {k: v.numpy() for k, v in host.items()}
    tmp = np.empty(5 * arr["key"].size, np.float32)
    out = np.empty_like(arr["key"])
    for _ in range(warmup):
        c_port.chain_nq(arr["mv"], arr["key"], arr["scale_map"], arr["cur"], arr["logits"], tmp=tmp, out=out)
    t0 = time.perf_counter()
    for _ in range(reps):
        c_port.chain_nq(arr["mv"], arr["key"], arr["scale_map"], arr["cur"], arr["logits"], tmp=tmp, out=out)
    dt = time.perf_counter() - t0
    return sample_frames * reps / dt, c_port.num_threads(), 1e3 * dt / reps


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    # size the per-step sample so that warmup + K steps stay within a few minutes whatever K is
    probe_fps, _, _ = cpu_reference_fps(8, reps=1, warmup=1)
    budget_s = 150.0
    sample = int(max(1, min(8, budget_s * probe_fps / max(1, args.steps))))
    fps, cores, ms = cpu_reference_fps(sample, reps=max(1, args.steps), warmup=max(1, min(args.warmup, 3)))
    line = {
        "impl": "reference", "metric": METRIC, "value": fps, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(FRAMES_PER_GPU, args.gpus),      # the same dict as our arm's: same workload
        "cpu_baseline": {"value": fps, "unit": UNIT, "cores": cores, "kind": "port",
                         "sample": "each reference step is a bounded sample of %d frames of the workload, x %d steps; C port of "
                                   "the MXNet CPU operators (GridGenerator, BilinearSampler, mul, softmax, tile, mul, add), "
                                   "OpenMP" % (sample, args.steps)},
        "e2e": {"value": fps, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)
    return 0


# --------------------------------------------------------------------------------------------
# our arm
# --------------------------------------------------------------------------------------------
def measured_hbm_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return FALLBACK_HBM_GBS, "fallback (B200_PROFILING.md 6.65 TB/s)"


def recorded_traffic(frames):
    """dram bytes per launch of the dominant kernel from the committed ncu --set full capture (a RECORDED figure: a
    profiler cannot run inside the timed bench).  Returns (bytes per launch, pre-pass microseconds, source)."""
    try:
        with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as f:
            t = json.load(f)
        k = t["agg_nchw_tma_kernel"]
        return float(k["dram_bytes_per_frame"]) * frames, k.get("prepass_us"), \
            "recorded: profiles/ncu_traffic.json (%s)" % k.get("source", "ncu --set full of this kernel on this workload")
    except Exception:
        return None, None, "unavailable"


def measure_pinned_copy_peak(dev, world, barrier, gather, mb=192, reps=6):
    """GB/s of plain pinned-memory copies on every rank at once (whole-job aggregate, max time over ranks):
    H2D alone, D2H alone, and both directions concurrently with 3 bytes in per byte out (the e2e workload's ratio)."""
    import torch
    n = mb << 20
    h_in, h_out = torch.empty(3 * n, dtype=torch.uint8).pin_memory(), torch.empty(n, dtype=torch.uint8).pin_memory()
    d_in, d_out = torch.empty(3 * n, dtype=torch.uint8, device=dev), torch.empty(n, dtype=torch.uint8, device=dev)
    s1, s2 = torch.cuda.Stream(dev), torch.cuda.Stream(dev)
    cur = torch.cuda.current_stream()

    def run(do_in, do_out):
        for it in range(2):                       # pass 0 warms up, pass 1 is timed
            barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(cur)
            s1.wait_event(e0)
            s2.wait_event(e0)
            for _ in range(reps):
                if do_in:
                    with torch.cuda.stream(s1):
                        d_in.copy_(h_in, non_blocking=True)
                if do_out:
                    with torch.cuda.stream(s2):
                        h_out.copy_(d_out, non_blocking=True)
            cur.wait_stream(s1)
            cur.wait_stream(s2)
            e1.record(cur)
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1)
        nbytes = reps * ((3 * n if do_in else 0) + (n if do_out else 0))
        tot, max_ms = gather(nbytes, ms)
        return tot / (max_ms / 1e3) / 1e9

    out = {"h2d_gbs": run(True, False), "d2h_gbs": run(False, True), "mix_gbs": run(True, True)}
    del h_in, h_out, d_in, d_out
    return out


def run_ours(args):
    import torch
    import torch.distributed as dist

    from lsfa_b200 import _cabi, ops
    from lsfa_b200.host import HostAggregator
    from lsfa_b200.streams import gather_frame_counts

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device; there is no CPU fallback (use --impl reference for the CPU baseline)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    _cabi.load()
    frames = args.frames
    K, Wm = args.steps, max(args.warmup, 3)

    # one process per GPU: stay on the CPUs (and memory) of the GPU's NUMA node before any pinned buffer is allocated
    from lsfa_b200.host import bind_near_gpu
    affinity0 = os.sched_getaffinity(0)
    numa = bind_near_gpu(local) if os.environ.get("LSFA_BENCH_NO_NUMA_BIND") is None else {"bound": False, "skipped": True}
    host = make_host_inputs(frames, seed=1000 + rank)
    d = {k: v.to(dev, non_blocking=True) for k, v in host.items()}
    torch.cuda.synchronize()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---------------- value: inputs resident in HBM, one fused launch per step ----------------
    prep = ops.PreparedAggregate(d["key"], d["mv"], flow_kind="raw", cur=d["cur"], scale_map=d["scale_map"],
                                 weight_mode="logits", logits=d["logits"])
    stream = torch.cuda.current_stream().cuda_stream
    for _ in range(Wm):
        prep.run(stream)
    barrier()
    sampler = ClockSampler(local)
    sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(K):
        prep.run(stream)
    e1.record()
    barrier()
    sampler.stop()
    ms_local = e0.elapsed_time(e1)
    total_frames, ms = gather_frame_counts(frames * K, ms_local)
    value = total_frames / (ms / 1e3)
    launches = K * prep.launches
    clocks = sampler.summary()
    dumps = {} if args.dump_outputs is not None and rank == 0 else None
    if dumps is not None:
        dumps["value"] = dump_sample(prep.out)

    # roofline of the dominant (only) kernel: algorithmic bytes per launch / launch duration
    peak, peak_src = measured_hbm_peak()
    alg_bytes = algorithmic_bytes_v2(frames)
    launch_ms = ms_local / K
    achieved = alg_bytes / (launch_ms / 1e3) / 1e9
    traffic, prepass_us, traffic_src = recorded_traffic(frames)
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": traffic, "traffic_source": traffic_src, "kernel": "agg_nchw_tma_kernel<K=2,PPT=5,ScaleCur>",
                "prepass_us_recorded": prepass_us,
                "note": "launch_ms is one whole step = agg_records_kernel (index-math pre-pass: 11-12 us in the ncu launch "
                        "list under profiles/, ~3 % of the step) + the dominant streaming kernel, so `achieved` understates "
                        "the dominant kernel on its own by that share. `peak` is "
                        "the driver-measured torch copy bandwidth (MEASURED_PEAKS.json: b.copy_(a), 1 Gi bf16), not the "
                        "hardware limit: a TMA-in/TMA-out kernel whose traffic is 3/4 reads can exceed it (frac > 1); "
                        "frac_of_nominal_8TBs and ncu's dram__throughput (profiles/) are the conservative views",
                "algorithmic_bytes_per_launch": alg_bytes, "launch_ms": launch_ms, "peak_source": peak_src,
                "frac_of_nominal_8TBs": achieved / 8000.0}

    # ---------------- e2e: host buffers in, host buffer out, copies inside the timed region ----
    # (a) what the box can move: a plain pinned cudaMemcpyAsync loop on ALL ranks at once, H2D and D2H concurrently in the
    #     workload's own byte ratio - the denominator of e2e.roofline
    copy_peak = measure_pinned_copy_peak(dev, world, barrier, gather_frame_counts)
    # (b) the reference-facing call: one C-ABI lsfa_host_aggregate_f32_nchw per 64-frame batch (lsfa_b200.host.HostAggregator)
    agg = HostAggregator(frames, C, H, W, (MV_H, MV_W), dev, chunk=args.chunk, depth=3)
    out_host = torch.empty((frames, C, H, W), dtype=torch.float32).pin_memory()
    e2e_steps = K if args.e2e_steps <= 0 else args.e2e_steps

    def time_host_path(agg_, host_, steps):
        for _ in range(3):
            agg_(host_, out_host)
        agg_.synchronize()
        barrier()
        agg_.launches = 0
        cur_stream = torch.cuda.current_stream()
        pipe_streams = (agg_.s_in, agg_.s_run, agg_.s_out)
        f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        f0.record(cur_stream)
        for s_ in pipe_streams:
            s_.wait_event(f0)                 # the pipeline starts after the start mark ...
        for _ in range(steps):
            agg_(host_, out_host)
        for s_ in pipe_streams:
            cur_stream.wait_stream(s_)        # ... and the stop mark waits for every copy and kernel
        f1.record(cur_stream)
        agg_.synchronize()
        torch.cuda.synchronize()
        ms_l = f0.elapsed_time(f1)
        barrier()
        return gather_frame_counts(frames * steps, ms_l)

    e2e_frames, e2e_ms = time_host_path(agg, host, e2e_steps)
    if dumps is not None:
        dumps["e2e"] = dump_sample(out_host)
    bi, bo = agg.bytes_per_call()
    e2e_gbs = world * (bi + bo) * e2e_steps / (e2e_ms / 1e3) / 1e9
    e2e = {"value": e2e_frames / (e2e_ms / 1e3), "unit": UNIT, "h2d_bytes_per_step": bi, "d2h_bytes_per_step": bo,
           "steps": e2e_steps, "ms_per_step": e2e_ms / e2e_steps, "launches_per_step": agg.launches // max(1, e2e_steps),
           "host_numa_binding_rank0": numa,
           "roofline": {"bound": "pcie", "achieved": e2e_gbs, "peak": copy_peak["mix_gbs"], "unit": "GB/s",
                        "frac": e2e_gbs / copy_peak["mix_gbs"] if copy_peak["mix_gbs"] else None,
                        "peak_source": "measured in this run: pinned cudaMemcpyAsync loop, H2D and D2H concurrently (3:1 bytes, "
                                       "the workload's ratio) on all %d rank(s) at once, whole-job GB/s" % world,
                        "h2d_only_gbs": copy_peak["h2d_gbs"], "d2h_only_gbs": copy_peak["d2h_gbs"]},
           "api": "lsfa_host_aggregate_f32_nchw through lsfa_b200.host.HostAggregator (one C-ABI call per batch: pinned host "
                  "in/out, %d-frame chunks, 3-stream pipeline over caller-owned staging; of each 600x1000 MV field only the 2 "
                  "rows in 16 the reference's stride-16 resize reads cross PCIe)" % agg.chunk}
    checksum_src = out_host[0, 0, 0, :8].clone()
    # (c) the reference's GOP contract (core/tester.py:246-252): key feature resident on the device, one upload per GOP of
    #     11 non-key frames; every frame still brings its own scale map, current feature, MVs and logits and takes its output home
    gop_len = 11
    n_keys = (frames + gop_len - 1) // gop_len
    agg_g = HostAggregator(frames, C, H, W, (MV_H, MV_W), dev, chunk=args.chunk, depth=3, num_slots=n_keys)
    host_g = {k: host[k] for k in ("scale_map", "cur", "mv", "logits")}
    host_g["key_index"] = (torch.arange(frames, dtype=torch.int32) // gop_len).pin_memory()
    host_g["new_keys"] = host["key"][:n_keys]
    host_g["key_slot"] = torch.arange(n_keys, dtype=torch.int32).pin_memory()
    g_frames, g_ms = time_host_path(agg_g, host_g, e2e_steps)
    if dumps is not None:
        dumps["e2e_gop"] = dump_sample(out_host)
    gbi, gbo = agg_g.bytes_per_call(host_g)
    g_gbs = world * (gbi + gbo) * e2e_steps / (g_ms / 1e3) / 1e9
    e2e["gop_contract"] = {"value": g_frames / (g_ms / 1e3), "unit": UNIT, "h2d_bytes_per_step": gbi, "d2h_bytes_per_step": gbo,
                           "ms_per_step": g_ms / e2e_steps, "key_uploads_per_step": n_keys, "gop_len": gop_len,
                           "achieved_gbs": g_gbs, "frac_of_measured_copy_peak": g_gbs / copy_peak["mix_gbs"] if copy_peak["mix_gbs"] else None,
                           "note": "second row, not the headline: the key feature stays in a device table across its GOP "
                                   "(core/tester.py:246-252), frames name their slot through key_index"}
    del agg_g
    checksum = float(checksum_src.sum())    # the result really is on the host
    try:
        os.sched_setaffinity(0, affinity0)           # the CPU baseline below gets every host core back
    except OSError:
        pass

    extra = {}
    if rank == 0 and not args.no_extra:
        extra = run_extras(dev, d, args)

    cpu_baseline = None
    if rank == 0 and not args.no_cpu_baseline:
        try:
            fps1, cores, _ = cpu_reference_fps(8, reps=1, warmup=1)
            budget = 15.0 if world == 1 else 4.0      # N > 1: a short sample, the other ranks wait at the final barrier
            reps = int(max(2, min(800, budget / max(8 / fps1, 1e-3))))     # ~15 s of CPU work
            fps, cores, _ = cpu_reference_fps(8, reps=reps, warmup=0)
            cpu_baseline = {"value": fps, "unit": UNIT, "cores": cores, "kind": "port",
                            "sample": "8 frames x %d repetitions (~%.0f s) of the same workload; C port of the MXNet "
                                      "CPU operator chain, OpenMP over all host threads" % (reps, reps * 8 / fps)}
        except Exception as e:  # the baseline must never take the GPU result down with it
            cpu_baseline = {"value": None, "unit": UNIT, "cores": 0, "kind": "port", "sample": "failed: %r" % (e,)}

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": Wm,
            "ms_per_step": ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": workload_config(frames, world),
            "roofline": roofline, "cpu_baseline": cpu_baseline, "e2e": e2e, "gpu_launches": launches,
            "clocks": clocks, "achieved_hbm_gbs_per_gpu": achieved, "host_checksum": checksum,
        }
        if extra:
            line["extra"] = extra
        if dumps is not None:
            import numpy as np
            os.makedirs(args.dump_outputs, exist_ok=True)
            for name, a in dumps.items():
                np.save(os.path.join(args.dump_outputs, name + ".npy"), a)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()
    return 0


def time_launches(fn, warmup, steps):
    import torch
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def run_extras(dev, d, args):
    """Secondary numbers (never the headline): bf16 NHWC variant, unfused ablation, hi-res config.  They time their own
    step counts (--steps capped at 20, or fixed per row), recorded as each row's "steps"."""
    import torch

    from lsfa_b200 import ops
    out = {}
    peak, _ = measured_hbm_peak()
    frames = d["key"].shape[0]
    steps = min(args.steps, 20)
    try:
        # unfused reference graph (9 kernels, 16F of traffic) vs fused, same fp32 inputs
        flow = ops.mv_pool(d["mv"])
        tmp = torch.empty(5 * d["key"].numel(), dtype=torch.float32, device=dev)
        ms_u = time_launches(lambda: ops.unfused_chain(d["key"], flow, d["scale_map"], d["cur"], d["logits"], tmp), 3, steps)
        out["unfused_fp32_nchw"] = {"frames_per_s": frames / (ms_u / 1e3), "ms_per_step": ms_u, "launches_per_step": 9,
                                    "steps": steps}
        del tmp
    except Exception as e:
        out["unfused_fp32_nchw"] = {"error": repr(e)}
    try:
        # the LDG/STG plane-resident kernel (previous headline) on the same inputs
        prep2 = ops.PreparedAggregate(d["key"], d["mv"], flow_kind="raw", cur=d["cur"], scale_map=d["scale_map"],
                                      weight_mode="logits", logits=d["logits"], force_generic=2)
        s2 = torch.cuda.current_stream().cuda_stream
        ms_p = time_launches(lambda: prep2.run(s2), 3, steps)
        gb = algorithmic_bytes_v2(frames, 4) / (ms_p / 1e3) / 1e9
        out["fused_fp32_nchw_plane_ldg"] = {"frames_per_s": frames / (ms_p / 1e3), "ms_per_step": ms_p,
                                            "achieved_gbs": gb, "frac_of_measured_peak": gb / peak, "steps": steps}
    except Exception as e:
        out["fused_fp32_nchw_plane_ldg"] = {"error": repr(e)}
    try:
        # config 3 shape: bf16 NHWC (batch limited by what is already resident: same frame count)
        nh = {k: ops.to_nhwc(d[k], torch.bfloat16) for k in ("key", "cur", "scale_map")}
        prep = ops.PreparedAggregate(nh["key"], d["mv"], flow_kind="raw", cur=nh["cur"], scale_map=nh["scale_map"],
                                     weight_mode="logits", logits=d["logits"], layout="nhwc_bf16")
        s = torch.cuda.current_stream().cuda_stream
        ms_b = time_launches(lambda: prep.run(s), 3, steps)
        gb = algorithmic_bytes_v2(frames, 2) / (ms_b / 1e3) / 1e9
        out["fused_bf16_nhwc"] = {"frames_per_s": frames / (ms_b / 1e3), "ms_per_step": ms_b, "achieved_gbs": gb,
                                  "frac_of_measured_peak": gb / peak, "steps": steps}
        # BASELINE configs[2] proper: the same in bf16 channels-last at batch 512 (the resident frames tiled 512/frames times)
        reps = max(1, 512 // frames)
        if reps > 1:
            big = {k: v.repeat(reps, 1, 1, 1) for k, v in nh.items()}
            prep = ops.PreparedAggregate(big["key"], d["mv"].repeat(reps, 1, 1, 1), flow_kind="raw", cur=big["cur"],
                                         scale_map=big["scale_map"], weight_mode="logits",
                                         logits=d["logits"].repeat(reps, 1, 1, 1), layout="nhwc_bf16")
            ms_c = time_launches(lambda: prep.run(s), 3, min(steps, 10))
            nb = frames * reps
            gb = algorithmic_bytes_v2(nb, 2) / (ms_c / 1e3) / 1e9
            out["fused_bf16_nhwc_batch512"] = {"frames": nb, "frames_per_s": nb / (ms_c / 1e3), "ms_per_step": ms_c,
                                               "achieved_gbs": gb, "frac_of_measured_peak": gb / peak, "steps": min(steps, 10)}
            del big, prep
        nf = {k: ops.to_nhwc(d[k], torch.float32) for k in ("key", "cur", "scale_map")}
        prep = ops.PreparedAggregate(nf["key"], d["mv"], flow_kind="raw", cur=nf["cur"], scale_map=nf["scale_map"],
                                     weight_mode="logits", logits=d["logits"], layout="nhwc_f32")
        ms_f = time_launches(lambda: prep.run(s), 3, steps)
        gb = algorithmic_bytes_v2(frames, 4) / (ms_f / 1e3) / 1e9
        out["fused_fp32_nhwc"] = {"frames_per_s": frames / (ms_f / 1e3), "ms_per_step": ms_f, "achieved_gbs": gb,
                                  "frac_of_measured_peak": gb / peak, "steps": steps}
    except Exception as e:
        out["fused_bf16_nhwc"] = {"error": repr(e)}
    for name, fn in (("cfg1_single_frame", extra_cfg1), ("cfg4_hires_68x120", extra_cfg4), ("cfg5_multi_stream", extra_cfg5),
                     ("keyframe_networks_tcgen05", extra_keyframe), ("backward_training_path", extra_backward)):
        torch.cuda.empty_cache()
        try:
            out[name] = fn(dev, d, peak, steps)
        except Exception as e:
            out[name] = {"error": repr(e)}
    return out


def extra_cfg1(dev, d, peak, steps):
    """BASELINE configs[0]: ONE non-key frame, 1024x38x63 fp32 + a 600x1000 MV field, GridGenerator(warp) + BilinearSampler:
    latency of the three drop-in operators and of the fused op (eager and replayed from a CUDA graph), with the stronger
    CPU baseline SURVEY 8d names beside it: torch.nn.functional.grid_sample on the host's cores."""
    import torch

    from lsfa_b200 import ops
    F4, HW = C * H * W * 4, H * W
    key, mv = d["key"][:1].contiguous(), d["mv"][:1].contiguous()
    s = torch.cuda.current_stream().cuda_stream
    grid = torch.empty((1, 2, H, W), device=dev)
    o = torch.empty_like(key)
    r = {"steps": 200}                  # per timing below
    ms = time_launches(lambda: ops.BilinearSampler(key, ops.GridGenerator(ops.mv_pool(mv), out=grid), out=o), 10, 200)
    r["three_dropin_operators_us"] = 1e3 * ms
    p0 = ops.PreparedAggregate(key, mv, flow_kind="raw")
    ms = time_launches(lambda: p0.run(s), 10, 200)
    r["fused_warp_us"] = 1e3 * ms
    r["fused_warp_launches"] = p0.launches
    p2 = ops.PreparedAggregate(key, mv, flow_kind="raw", cur=d["cur"][:1].contiguous(), scale_map=d["scale_map"][:1].contiguous(),
                               weight_mode="logits", logits=d["logits"][:1].contiguous())
    ms = time_launches(lambda: p2.run(s), 10, 200)
    r["fused_v2_us"] = 1e3 * ms
    r["fused_v2_launches"] = p2.launches
    for tag, p in (("fused_warp_graph_us", p0), ("fused_v2_graph_us", p2)):
        # recorded and replayed through the C ABI (lsfa_graph_begin / _end / _launch), not through torch
        side = torch.cuda.Stream()
        with torch.cuda.stream(side):
            for _ in range(3):
                p.run(side.cuda_stream)
            side.synchronize()
            g = ops.RecordedGraph(side.cuda_stream)
            with g:
                p.run(side.cuda_stream)
        r[tag] = 1e3 * time_launches(lambda: g.launch(s), 10, 200)
        g.close()
    r["graph_api"] = "lsfa_graph_begin / lsfa_graph_end / lsfa_graph_launch (C ABI)"
    r["bytes_v0"] = 2 * F4 + 32 * HW
    r["frac_of_measured_peak_fused_warp_graph"] = r["bytes_v0"] / (r["fused_warp_graph_us"] * 1e-6) / 1e9 / peak
    # CPU side by side: torch.grid_sample (align_corners=True, zeros) = a7+a8 on the host cores
    try:
        nthr = len(os.sched_getaffinity(0))
        torch.set_num_threads(nthr)
        kc = key.cpu()
        gc = ops.GridGenerator(ops.mv_pool(mv)).cpu().permute(0, 2, 3, 1).contiguous()
        for _ in range(3):
            torch.nn.functional.grid_sample(kc, gc, mode="bilinear", padding_mode="zeros", align_corners=True)
        t0 = time.perf_counter()
        for _ in range(10):
            torch.nn.functional.grid_sample(kc, gc, mode="bilinear", padding_mode="zeros", align_corners=True)
        r["cpu_torch_grid_sample_ms"] = 1e3 * (time.perf_counter() - t0) / 10
        r["cpu_threads"] = nthr
    except Exception as e:
        r["cpu_torch_grid_sample_ms"] = None
        r["cpu_error"] = repr(e)
    return r


def extra_cfg4(dev, d, peak, steps):
    """BASELINE configs[3]: 1080p -> 1024x68x120 features, batch 128, fused V2 in fp32 NCHW and bf16 channels-last
    (inputs generated on the device; 17 GB / 8.6 GB working sets)."""
    import torch

    from lsfa_b200 import ops
    N4, H4, W4 = 128, 68, 120
    g = torch.Generator(device=dev).manual_seed(4)
    blk = torch.randint(-96, 97, (N4, H4, W4, 2), device=dev, generator=g, dtype=torch.int32)
    blk[torch.rand((N4, H4, W4), device=dev, generator=g) < 0.5] = 0
    mv = blk.repeat_interleave(16, 1).repeat_interleave(16, 2)[:, :1080, :1920].contiguous()
    lg = torch.randn((N4, 2, H4, W4), device=dev, generator=g)
    r = {}
    s = torch.cuda.current_stream().cuda_stream
    for tag, dt, lay, fb in (("fp32_nchw", torch.float32, "nchw", 4), ("bf16_nhwc", torch.bfloat16, "nhwc_bf16", 2)):
        shape = (N4, C, H4, W4) if lay == "nchw" else (N4, H4, W4, C)
        key = torch.randn(shape, device=dev, generator=g, dtype=torch.float32).clamp_(min=0).to(dt)
        cur = torch.randn(shape, device=dev, generator=g, dtype=torch.float32).clamp_(min=0).to(dt)
        sm = (1 + 0.1 * torch.randn(shape, device=dev, generator=g, dtype=torch.float32)).to(dt)
        prep = ops.PreparedAggregate(key, mv, flow_kind="raw", cur=cur, scale_map=sm, weight_mode="logits", logits=lg, layout=lay)
        ms = time_launches(lambda: prep.run(s), 3, min(steps, 10))
        alg = N4 * (4 * C * H4 * W4 * fb + 40 * H4 * W4)
        gb = alg / (ms / 1e3) / 1e9
        r[tag] = {"frames": N4, "frames_per_s": N4 / (ms / 1e3), "ms_per_step": ms, "achieved_gbs": gb, "frac_of_measured_peak": gb / peak,
                  "steps": min(steps, 10)}
        del key, cur, sm, prep
        torch.cuda.empty_cache()
    return r


def extra_cfg5(dev, d, peak, steps):
    """BASELINE configs[4] on this GPU: 256 independent streams x 10 non-key frames through lsfa_b200.driver.StreamScheduler
    (one key feature per stream in a device table, frames name it through key_index; the reference's shipped non-key graph
    SYM:570-586: warp(key, MV) + rnet_conv0(res) + current feature).  tools/bench_streams.py sweeps 64..1024 streams."""
    import torch

    from lsfa_b200 import streams
    from lsfa_b200.driver import StreamScheduler
    S, B = 256, 80
    g = torch.Generator(device=dev).manual_seed(5)
    cur = d["cur"][:min(B, d["cur"].shape[0])]
    reps = -(-B // cur.shape[0])
    cur = cur.repeat(reps, 1, 1, 1)[:B].contiguous()
    mv = d["mv"].repeat(reps, 1, 1, 1)[:B].contiguous()
    res = torch.randn((B, 3, H, W), device=dev, generator=g) * 30
    rnet_w = 0.01 * torch.randn((C, 3), device=dev, generator=g)
    rnet_b = torch.zeros((C,), device=dev)
    out = torch.empty_like(cur)
    sch = StreamScheduler([streams.KEY_FRAME_INTERVAL] * S, C, (H, W), dev)
    sch.key_table.normal_(generator=g).clamp_(min=0)
    batches = sch.batches(B)
    slots = [torch.as_tensor(b[2], dtype=torch.int32, device=dev) for b in batches]
    frames = sum(len(b[2]) for b in batches)

    def step():
        for sl in slots:
            m = sl.numel()
            sch.run_non_key_batch(sl, mv[:m], cur[:m], res=res[:m], rnet_w=rnet_w, rnet_b=rnet_b, out=out[:m])

    ms = time_launches(step, 2, 5)
    F4, HW = C * H * W * 4, H * W
    alg = 2 * F4 + F4 // 10 + 44 * HW
    fps = frames / (ms / 1e3)
    return {"streams": S, "frames_per_step": frames, "launches_per_step": len(slots), "ms_per_step": ms, "frames_per_s": fps,
            "alg_bytes_per_frame": alg, "achieved_gbs": fps * alg / 1e9, "frac_of_measured_peak": fps * alg / 1e9 / peak,
            "key_table_gb": sch.key_table.numel() * 4 / 1e9, "steps": 5}


def extra_backward(dev, d, peak, steps):
    """SURVEY 8f rank 4 (get_train_symbol SYM:306-338): backward of GridGenerator(warp)+BilinearSampler as a gather
    (deterministic d/d(key)), and of the fused operator with its tails, 64 frames of 1024x38x63 fp32; algorithmic bytes =
    every stream once (3F / 2F for the sampler, 10F for the fused V2 backward incl. its d/d(warp) intermediate)."""
    import torch

    from lsfa_b200 import ops
    F4, HW = C * H * W * 4, H * W
    n = d["key"].shape[0]
    flow = ops.mv_pool(d["mv"])
    og = torch.randn_like(d["key"])
    gk, gf = torch.empty_like(d["key"]), torch.empty_like(flow)
    ws = torch.empty(ops.A.load().lsfa_bilinear_sampler_backward_workspace_bytes(n, C, H, W, H, W), dtype=torch.uint8, device=dev)
    r = {"frames": n}
    for tag, fn, alg in (
            ("warp_backward_key_and_flow", lambda: ops.warp_backward(d["key"], flow, og, grad_key=gk, grad_flow=gf, workspace=ws, kernel="gather"), 3 * F4 + 16 * HW),
            ("warp_backward_key_only", lambda: ops.warp_backward(d["key"], flow, og, grad_key=gk, req_flow="null", workspace=ws, kernel="gather"), 2 * F4 + 8 * HW),
            ("fused_v2_backward_all_gradients", lambda: ops.warp_scale_aggregate_backward(og, d["key"], flow, flow_kind="flow", cur=d["cur"], scale_map=d["scale_map"], weight_mode="logits", logits=d["logits"]), 10 * F4)):
        ms = time_launches(fn, 2, 10)
        gb = n * alg / (ms / 1e3) / 1e9
        r[tag] = {"ms_per_step": ms, "frames_per_s": n / (ms / 1e3), "achieved_gbs": gb, "frac_of_measured_peak": gb / peak, "steps": 10}
    return r


def extra_keyframe(dev, d, peak, steps):
    """SURVEY 8f rank 2: the embedding network + cosine logits of Fgfa_net and the Nq network (SYM:94-139) for 16 key frames at
    1024x38x63: this package's tcgen05 implicit-GEMM kernels against cuDNN's bf16 channels-last convolutions on the same
    operands, with the fraction of the measured sustained bf16 tensor peak."""
    import torch

    from lsfa_b200 import graphs, ops
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            tf_peak = float(json.load(f)["bf16_tflops_sustained"])
        tf_src = "measured (MEASURED_PEAKS.json bf16_tflops_sustained)"
    except Exception:
        tf_peak, tf_src = 1400.0, "fallback (B200_PROFILING.md ~1.4 PFLOP/s sustained)"
    N, E = 16, 2048
    HW = H * W
    g = torch.Generator(device=dev).manual_seed(6)
    rn = lambda *sh: 0.01 * torch.randn(sh, device=dev, generator=g)  # noqa: E731
    emb = (rn(512, C, 1, 1), rn(512), rn(512, 512, 3, 3), rn(512), rn(E, 512, 1, 1), rn(E))
    nq = (rn(256, C, 3, 3), rn(256), rn(16, 256, 1, 1), rn(16), rn(1, 16, 1, 1), rn(1))
    x = torch.cat([d["cur"][:N], d["key"][:N]], dim=0)
    xb = graphs._lowp_input([x], torch.bfloat16)                  # logical NCHW, channels-last bf16
    xn = xb.permute(0, 2, 3, 1)
    gf_emb = 2 * N * 2 * HW * (C * 512 + 9 * 512 * 512 + 512 * E) / 1e9
    gf_nq = 2 * N * 2 * HW * (9 * C * 256 + 256 * 16 + 16) / 1e9
    pe, pq = graphs.pack_embed_params(emb), graphs.pack_nq_params(nq)
    embb, nqb = graphs.prepare_params(emb, torch.bfloat16), graphs.prepare_params(nq, torch.bfloat16)
    r = {"key_frames": N, "tensor_peak_tflops": tf_peak, "tensor_peak_source": tf_src}
    ms = time_launches(lambda: ops.embed_cosine_logits(xn, pe), 3, 10)
    r["embed_cosine_tcgen05"] = {"ms": ms, "gflop": gf_emb, "tflops": gf_emb / ms, "frac_of_sustained_bf16_peak": gf_emb / ms / tf_peak,
                                 "launches": 4, "writes_embeddings": False, "steps": 10}
    ms = time_launches(lambda: ops.nq_logits(xn, pq), 3, 10)
    r["nq_tcgen05"] = {"ms": ms, "gflop": gf_nq, "tflops": gf_nq / ms, "frac_of_sustained_bf16_peak": gf_nq / ms / tf_peak, "launches": 1,
                       "steps": 10}
    ms = time_launches(lambda: graphs.embed_net(xb, *embb), 2, 5)
    r["embed_convs_cudnn_bf16"] = {"ms": ms, "tflops": gf_emb / ms, "note": "library arm: convolutions only, embeddings written to HBM, cosine not included",
                                   "steps": 5}
    ms = time_launches(lambda: graphs.nq_net(xb, *nqb), 2, 5)
    r["nq_convs_cudnn_bf16"] = {"ms": ms, "tflops": gf_nq / ms, "steps": 5}
    return r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--frames", type=int, default=FRAMES_PER_GPU, help="frames per GPU per step")
    ap.add_argument("--chunk", type=int, default=8, help="frames per H2D/D2H pipeline chunk (e2e)")
    ap.add_argument("--e2e-steps", type=int, default=0, help="0 = same as --steps")
    ap.add_argument("--no-extra", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the last timed step's outputs as DIR/<name>.npy (float32, sampled; --impl ours, rank 0)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        return run_reference(args)
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
