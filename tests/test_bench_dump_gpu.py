"""GPU: bench.py --dump-outputs writes what the timed path returned for its last timed step - checked against an eager
forward of that same step (same seeds, same sampler RNG counter, same weights)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import ROOT, rel_err

pytestmark = pytest.mark.gpu


def test_dump_outputs_is_the_last_timed_step(tmp_path):
    steps, warmup = 3, 2
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", str(steps), "--warmup", str(warmup),
                        "--cpu-batches", "0", "--no-config3", "--math", "tf32x3", "--dump-outputs", str(tmp_path)],
                       cwd=ROOT, stdout=subprocess.PIPE, stderr=subprocess.PIPE, timeout=900)
    assert p.returncode == 0, p.stderr.decode()[-2000:]
    lines = [ln for ln in p.stdout.decode().splitlines() if ln.startswith("{")]
    assert len(lines) == 1 and json.loads(lines[0])["steps"] == steps
    got = np.load(tmp_path / "embeddings.npy")

    import bench
    import graphsage_b200 as gs
    assert got.dtype == np.float32 and got.shape == (bench.BATCH, 2 * bench.DIM)
    g = bench.build_graph()
    table = torch.zeros((bench.N_NODES + 1, gs.ops.pad_cols(bench.F)), dtype=torch.float32, device="cuda")
    table[:, :bench.F] = torch.from_numpy(g["features"]).cuda()
    adj = torch.from_numpy(g["adj"]).cuda()
    gs.set_default_math("tf32x3")
    try:
        sampler = gs.UniformNeighborSampler(adj, seed=123)
        infos = [gs.SAGEInfo("node", sampler, bench.FANOUT[0], bench.DIM),
                 gs.SAGEInfo("node", sampler, bench.FANOUT[1], bench.DIM)]
        model = gs.SampleAndAggregate({"batch_size": bench.BATCH, "dropout": 0.}, table[:, :bench.F], adj, None, infos,
                                      concat=True, aggregator_type="mean")
        seeds = np.random.RandomState(1000).randint(0, bench.N_NODES, size=(warmup + steps, bench.BATCH)).astype(np.int32)
        model.forward(torch.from_numpy(seeds[0]))            # creates the aggregators, as bench.py's first forward does
        for a, w in zip(model.aggregators, bench.make_weights("mean", np.random.RandomState(7))):
            for k, v in w.items():
                a.vars[k] = torch.from_numpy(v).cuda()
        last = warmup + steps - 1
        # bench.py's pipeline continues the sampler's call count after that first forward: its step i draws what eager
        # forward number 1 + i draws
        sampler.counter = len(infos) * (1 + last)
        ref = model.forward(torch.from_numpy(seeds[last]), normalize=True).cpu().numpy()
    finally:
        gs.set_default_math("fp32")
    assert rel_err(got, ref) < 1e-4
