#!/usr/bin/env python
"""Check what ``bench.py --dump-outputs DIR`` wrote against the float64 reference (oracle/ref64.py), on the CPU.

  python tools/check_bench_outputs.py DIR [--frames 64]

value.npy (the headline PreparedAggregate), e2e.npy (HostAggregator, private keys) and e2e_gop.npy (the GOP form:
frame i samples key i // 11) are all the same operation on ``bench.make_host_inputs(frames, 1000)``: warp(key, raw MV)
x scale map, softmax-logit blend with the current feature.  Each file holds the values at the flat indices
``np.sort(default_rng(0).integers(0, numel, bench.DUMP_SAMPLE))`` (``bench.dump_sample``), or every value when the
output is smaller.  Prints one JSON line with the largest err/tol per file; exits 1 when any value is outside the gate.
"""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import bench  # noqa: E402
from oracle import ref64 as R  # noqa: E402

GOP_LEN = 11
FILES = ("value", "e2e", "e2e_gop")


def sample_index(numel):
    if numel <= bench.DUMP_SAMPLE:
        return np.arange(numel)
    return np.sort(np.random.default_rng(0).integers(0, numel, bench.DUMP_SAMPLE))


def reference_at(host, co, idx, key_index=None):
    """(ref, mag) float64 at the flat NCHW indices ``idx`` (sorted), frame chunk by frame chunk."""
    import torch
    N = host["key"].shape[0]
    per = host["key"][0].numel()
    ref, mag = np.empty(idx.size), np.empty(idx.size)
    for n0 in range(0, N, R.CHUNK):
        lo, hi = np.searchsorted(idx, [n0 * per, min(n0 + R.CHUNK, N) * per])
        if lo == hi:
            continue
        r, m = R.forward(host["key"], co, cur=host["cur"], scale_map=host["scale_map"], mode="logits",
                         logits=host["logits"], key_index=key_index, frames=range(n0, min(n0 + R.CHUNK, N)),
                         device=torch.device("cpu"))
        local = torch.from_numpy(idx[lo:hi] - n0 * per)
        ref[lo:hi] = r.flatten()[local].numpy()
        mag[lo:hi] = m.flatten()[local].numpy()
    return ref, mag


def main(argv=None):
    import torch
    ap = argparse.ArgumentParser()
    ap.add_argument("dir")
    ap.add_argument("--frames", type=int, default=bench.FRAMES_PER_GPU)
    args = ap.parse_args(argv)
    host = bench.make_host_inputs(args.frames, seed=1000, pinned=False)
    co = R.coords(mv=host["mv"])
    shape = (args.frames, bench.C, bench.H, bench.W)
    idx = sample_index(int(np.prod(shape)))
    result, ok = {}, True
    cache = {}
    for name in FILES:
        path = os.path.join(args.dir, name + ".npy")
        if not os.path.exists(path):
            result[name] = {"error": "missing"}
            ok = False
            continue
        got = np.load(path).reshape(-1).astype(np.float64)
        if got.size != idx.size:
            result[name] = {"error": "%d values, expected %d" % (got.size, idx.size)}
            ok = False
            continue
        ki = (np.arange(args.frames) // GOP_LEN).astype(np.int32) if name == "e2e_gop" else None
        if (ki is None) not in cache:                      # value and e2e compute the same thing
            cache[ki is None] = reference_at(host, co, idx, ki)
        ref, mag = cache[ki is None]
        tol = R.tolerance(torch.from_numpy(ref), torch.from_numpy(mag)).numpy()
        err = np.abs(got - ref)
        bad = ~(err <= tol)
        ratio = np.where(tol > 0, err / np.where(tol > 0, tol, 1.0), 0.0)
        entry = {"samples": int(idx.size), "max_err_over_tol": float(np.max(np.where(bad, np.inf, ratio)))}
        if bad.any():
            ok = False
            i = int(np.argmax(np.where(bad, np.nan_to_num(err - tol, nan=np.inf), -1.0)))
            entry.update(outside=int(bad.sum()), worst_nchw=[int(v) for v in np.unravel_index(idx[i], shape)],
                         got=float(got[i]), ref=float(ref[i]), tol=float(tol[i]))
        result[name] = entry
    print(json.dumps({"frames": args.frames, "gate": "|got-ref| <= %d u mag (oracle/ref64.py)" % R.K, "files": result,
                      "ok": ok}), flush=True)
    return 0 if ok else 1


if __name__ == "__main__":
    sys.exit(main())
