"""Cost of the LSTM aggregator (graphsage_seq) on the configs[1] workload: Reddit-shape graph (bench.build_graph), 2 hops,
fanout 25 x 10, batch 512, dims [602, 128, 128], concat, tf32x3 GEMMs, H = 128 ("small"); once with the fp32 feature
table and once with a bf16 table.

    python tools/seq_bench.py --out DIR [--steps 100 --warmup 20]

Prints one JSON line and writes it to DIR/seq_bench.json: per pass the CUDA-graph step time and seeds/s over an
event-timed region of --steps replays after --warmup, per-kernel event times (gather, projection GEMM, gs_lstm_seq, final
GEMM; a separate eager pass with per-launch events), the algorithmic FLOPs and bytes, and the GPU name, power limit and SM
clock read in the same run.  Needs a GPU; there is no CPU path."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.dont_write_bytecode = True
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

B, FAN, DIMS, H = 512, [25, 10], [602, 128, 128], 128


def algorithmic_cost():
    """FLOPs and bytes of one step from shapes (every sequence counted at its full fanout)."""
    seqs = {0: [(B, 10), (B * 10, 25)], 1: [(B, 10)]}           # layer -> [(sequences, k)] per hop
    fin = {0: DIMS[0], 1: 2 * DIMS[1]}
    proj = rec = final = 0
    gathered = pbytes = 0
    for layer, hops in seqs.items():
        for n, k in hops:
            proj += 2 * n * k * fin[layer] * 4 * H
            rec += 2 * n * k * H * 4 * H
            final += 2 * n * (fin[layer] + H) * DIMS[layer + 1]
            if layer == 0:
                gathered += 2 * n * k * fin[0] * 4                   # X written by the gather, read by the GEMM
            pbytes += 2 * n * k * 4 * H * 4                          # P written by the GEMM, read by gs_lstm_seq
    return {"projection_gflop": proj / 1e9, "recurrence_gflop": rec / 1e9, "final_gemm_gflop": final / 1e9,
            "gathered_x_bytes": gathered, "projection_p_bytes": pbytes}


def gpu_info():
    info = {"gpu": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader",
                            "-i", str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30)
        pl, sm, smax = [s.strip() for s in q.stdout.strip().split(",")]
        info.update(power_limit=pl, sm_clock=sm, sm_clock_max=smax)
    except Exception as e:                                         # reported, not guessed
        info.update(power_limit="unavailable (%s)" % e)
    return info


def run_pass(gs, g, table, steps, warmup):
    gs.set_default_math("tf32x3")
    adj = torch.from_numpy(g["adj"]).cuda()
    sampler = gs.UniformNeighborSampler(adj, seed=123)
    infos = [gs.SAGEInfo("node", sampler, FAN[0], DIMS[1]), gs.SAGEInfo("node", sampler, FAN[1], DIMS[2])]
    m = gs.SampleAndAggregate({"batch_size": B, "dropout": 0.}, table, adj, None, infos, concat=True,
                              aggregator_type="seq")
    rs = np.random.RandomState(7)
    pool = torch.from_numpy(rs.randint(0, g["n"], size=(64, B)).astype(np.int32)).cuda()
    # ---- per-kernel times: an eager pass with an event pair around every launch of ours
    for i in range(3):
        m.forward(pool[i])
    torch.cuda.synchronize()
    gs.ops.PROBE = {}
    reps = 5
    for i in range(reps):
        m.forward(pool[i])
    torch.cuda.synchronize()
    probe, gs.ops.PROBE = gs.ops.PROBE, None
    kern = {}
    for name, evs in probe.items():
        kern[name] = sum(a.elapsed_time(b) for a, b in evs) * 1e3 / reps      # us per step
    # gather launches carry no probe: time them with the profiler in the same eager setting
    from torch.autograd import DeviceType
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for i in range(reps):
            m.forward(pool[i])
        torch.cuda.synchronize()
    by_name = {}
    for e in prof.events():
        if e.device_type == DeviceType.CUDA:
            by_name[e.name] = by_name.get(e.name, 0.0) + e.time_range.elapsed_us() / reps
    gather_us = sum(v for k, v in by_name.items() if "gather_rows" in k)
    proj_rows = {B * 10, B * 10 * 25}                              # layer-0 / layer-1 projection GEMMs have M = n * k
    summary = {"gather_us": gather_us,
               "projection_gemm_us": sum(v for k, v in kern.items() if k.startswith("sage_gemm/")
                                         and int(k.split("/")[1]) in proj_rows),
               "lstm_seq_us": sum(v for k, v in kern.items() if k.startswith("lstm_seq/")),
               "final_gemm_us": sum(v for k, v in kern.items() if k.startswith("sage_gemm/")
                                    and int(k.split("/")[1]) in (B, B * 11)),
               "row_used_us": sum(v for k, v in kern.items() if k.startswith("row_used/")),
               "probes_us": {k: round(v, 2) for k, v in sorted(kern.items())},
               "profiler_kernels_us": {k: round(v, 2) for k, v in sorted(by_name.items())}}
    # ---- graphed step time
    sampler.counter = 0
    runner = m.graphed(B, normalize=True)
    for i in range(warmup):
        runner(pool[i % 64])
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(steps):
        runner(pool[i % 64])
    e1.record()
    torch.cuda.synchronize()
    step_us = e0.elapsed_time(e1) * 1e3 / steps
    runner.close()
    gs.set_default_math("fp32")
    return {"step_us": round(step_us, 2), "seeds_per_s": round(B / step_us * 1e6, 1), "launches_per_step":
            runner.launches_per_replay, "kernels": summary}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=20)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("seq_bench.py needs a CUDA device")
    import bench
    import graphsage_b200 as gs
    torch.cuda.set_device(0)
    info = gpu_info()
    g = bench.build_graph()
    table = torch.zeros((g["n"] + 1, gs.ops.pad_cols(602)), dtype=torch.float32, device="cuda")
    table[:, :602] = torch.from_numpy(g["features"]).cuda()
    res = {"workload": "reddit-shape N=%d F=602 graphsage_seq (H=%d) 2-hop fanout 25x10 batch %d dims %s concat tf32x3"
                       % (g["n"], H, B, DIMS),
           "timed_region": "%d CUDA-graph replays after %d warm-up replays" % (args.steps, args.warmup),
           "cost": algorithmic_cost()}
    res["fp32_table"] = run_pass(gs, g, table[:, :602], args.steps, args.warmup)
    tb = table.to(torch.bfloat16)
    res["bf16_table"] = run_pass(gs, g, tb[:, :602], args.steps, args.warmup)
    info2 = gpu_info()
    res.update(info)
    res["sm_clock_after"] = info2.get("sm_clock")
    os.makedirs(args.out, exist_ok=True)
    line = json.dumps(res)
    with open(os.path.join(args.out, "seq_bench.json"), "w") as fp:
        fp.write(line + "\n")
    print(line)


if __name__ == "__main__":
    main()
