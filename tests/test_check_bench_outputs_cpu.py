"""tools/check_bench_outputs.py on an oracle-made dump of bench.py's three outputs (2 frames: a sampled case)."""
import os
import sys

import numpy as np
import pytest
import torch

import bench
from oracle import lsfa_oracle as O

sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools"))
import check_bench_outputs as T  # noqa: E402

FRAMES = 2


@pytest.fixture(scope="module")
def dump(tmp_path_factory):
    d = tmp_path_factory.mktemp("dump")
    h = {k: v.numpy() for k, v in bench.make_host_inputs(FRAMES, seed=1000, pinned=False).items()}
    flow = O.mv_pool(h["mv"])
    for name, ki in (("value", None), ("e2e", None), ("e2e_gop", np.arange(FRAMES) // T.GOP_LEN)):
        out = O.warp_scale_aggregate(h["key"], flow, cur=h["cur"], scale_map=h["scale_map"], weight_mode=O.W_LOGITS,
                                     logits=h["logits"], key_index=ki)
        np.save(os.path.join(d, name + ".npy"), bench.dump_sample(torch.from_numpy(out)))
    return d


def test_oracle_dump_passes(dump, capsys):
    assert FRAMES * bench.C * bench.H * bench.W > bench.DUMP_SAMPLE          # the sampled path
    assert T.main([str(dump), "--frames", str(FRAMES)]) == 0
    assert '"ok": true' in capsys.readouterr().out


def test_one_perturbed_sample_fails(dump, tmp_path, capsys):
    for name in T.FILES:
        a = np.load(os.path.join(dump, name + ".npy"))
        if name == "e2e":
            i = int(np.argmax(np.abs(a) > 0.5))
            a[i] = np.float32(a[i] * (1 + 1e-4))
        np.save(os.path.join(tmp_path, name + ".npy"), a)
    assert T.main([str(tmp_path), "--frames", str(FRAMES)]) == 1
    out = capsys.readouterr().out
    assert '"ok": false' in out and '"outside": 1' in out
