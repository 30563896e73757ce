#!/usr/bin/env python
"""bench.py - seed nodes/sec through sample -> 2-hop gather -> aggregate (fanout 25x10) on a
Reddit-shaped synthetic graph (BASELINE.json configs[1]); one process per GPU.

    python bench.py --gpus 1 --steps 200 --warmup 20
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference --steps 5 --warmup 1      # the reference op sequence on host cores

A step = one 512-seed batch through the whole hot path.  Prints ONE JSON line (rank 0).  --dump-outputs DIR writes
the embeddings the timed path returned for its last step as DIR/embeddings.npy (float32), for comparing builds.
"""
import argparse
import json
import os
import sys
import threading
import time

import numpy as np
import torch

sys.dont_write_bytecode = True       # the tree may be read-only: leave it as it is
ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_NODES, F, MAX_DEG, BATCH, DIM = 232965, 602, 128, 512, 128
FANOUT = [25, 10]                    # layer order (samples_1, samples_2): hop-1 draws 10, hop-2 draws 25
ROWS_PER_BATCH = BATCH * (1 + 10 + 250)
GATHER_BYTES = ROWS_PER_BATCH * F * 4   # SURVEY 8(d): every gathered row counted once, no dedup credit


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler(threading.Thread):
    """Samples SM clock / throttle reasons through NVML while the timed region runs."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.stop_flag, self.max_mhz = index, [], set(), False, None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if self.nv is None:
            return
        nv = self.nv
        names = {nv.nvmlClocksEventReasonHwSlowdown if hasattr(nv, "nvmlClocksEventReasonHwSlowdown") else 0x8: "hw_slowdown",
                 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}
        while not self.stop_flag:
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h) if hasattr(nv, "nvmlDeviceGetCurrentClocksEventReasons") \
                    else nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.002)

    def summary(self):
        self.stop_flag = True
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["unavailable"]}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons)}


def build_graph(rank=0, world=1, barrier=None):
    """Reddit-shape synthetic graph (seed 123).  With several ranks, rank 0 generates it once and the
    others read it from /dev/shm (same bytes everywhere)."""
    from graphsage_b200.synthetic import reddit_like
    if world == 1:
        return reddit_like(n=N_NODES, f=F, max_degree=MAX_DEG, seed=123)
    base = "/dev/shm/gs_b200_graph_%d" % os.getuid()
    if rank == 0:
        g = reddit_like(n=N_NODES, f=F, max_degree=MAX_DEG, seed=123)
        np.save(base + "_adj.npy", g["adj"])
        np.save(base + "_feat.npy", g["features"])
        np.save(base + "_comm.npy", g["comm"])
        np.save(base + "_deg.npy", g["deg"])
    barrier()
    if rank != 0:
        g = dict(adj=np.load(base + "_adj.npy"), features=np.load(base + "_feat.npy"), comm=np.load(base + "_comm.npy"),
                 deg=np.load(base + "_deg.npy"), n=N_NODES, f=F, max_degree=MAX_DEG)
    barrier()
    if rank == 0:
        for suffix in ("_adj.npy", "_feat.npy", "_comm.npy", "_deg.npy"):
            os.remove(base + suffix)
    return g


def bench_config(workload, kind="mean"):
    """The same dict in both arms (the driver compares them): what is computed, not how."""
    return {"workload": workload, "batch": BATCH, "fanout": "25x10 (hop-1 draws 10, hop-2 draws 25)",
            "rows_gathered_per_step": ROWS_PER_BATCH, "feature_dtype": "bf16" if kind == "maxpool" else "f32",
            "l2": "inputs larger than L2 (567 MB feature table vs 126 MB L2; fresh random seeds every step)"}


def make_weights(kind, rs):
    """Random-init weights of the named architecture (glorot), shared by both arms."""
    def glorot(a, b):
        r = np.sqrt(6.0 / (a + b))
        return rs.uniform(-r, r, size=(a, b)).astype(np.float32)
    if kind == "mean":
        return [dict(neigh_weights=glorot(F, DIM), self_weights=glorot(F, DIM)),
                dict(neigh_weights=glorot(2 * DIM, DIM), self_weights=glorot(2 * DIM, DIM))]
    if kind == "gcn":
        return [dict(weights=glorot(F, 2 * DIM)), dict(weights=glorot(2 * DIM, 2 * DIM))]
    if kind == "maxpool":     # hidden 512 ("small"), reference graphsage/aggregators.py:139-142
        return [dict(mlp_weights=glorot(F, 512), mlp_bias=np.zeros(512, np.float32), neigh_weights=glorot(512, DIM),
                     self_weights=glorot(F, DIM)),
                dict(mlp_weights=glorot(2 * DIM, 512), mlp_bias=np.zeros(512, np.float32), neigh_weights=glorot(512, DIM),
                     self_weights=glorot(2 * DIM, DIM))]
    raise ValueError(kind)


def cpu_reference_rate(g, kind, weights, n_batches, warm, seed_rs, budget_s=None):
    """The reference op sequence on the host cores (oracle/torch_ref.py); seeds/s over n_batches.
    With budget_s, each step is a bounded sample (fewer seeds, same fanout) so the run fits the budget."""
    from oracle import torch_ref
    adj_t, feats_t = torch.from_numpy(g["adj"]), torch.from_numpy(g["features"])
    aggs = [{k: torch.from_numpy(v) for k, v in w.items()} for w in weights]
    concat = kind != "gcn"
    # use the thread count that is fastest on this host (all cores is often slower for the gather)
    ncpu = len(os.sched_getaffinity(0))
    best = (None, 1e30)
    probe_seeds = torch.from_numpy(np.random.RandomState(5).randint(0, N_NODES, size=BATCH).astype(np.int32))
    for nt in sorted({min(ncpu, t) for t in (8, 16, 32, 64, ncpu)}):
        torch.set_num_threads(nt)
        torch_ref.forward(adj_t, feats_t, probe_seeds, FANOUT, aggs, concat, kind, 123, 0, normalize=True)
        t0 = time.perf_counter()
        torch_ref.forward(adj_t, feats_t, probe_seeds, FANOUT, aggs, concat, kind, 123, 0, normalize=True)
        dt = time.perf_counter() - t0
        if dt < best[1]:
            best = (nt, dt)
    torch.set_num_threads(best[0])
    per_step = BATCH
    if budget_s is not None and best[1] * (warm + n_batches) > budget_s:
        per_step = int(max(16, min(BATCH, BATCH * budget_s / (best[1] * (warm + n_batches)))))
    cpu_reference_rate.per_step = per_step
    times = []
    for i in range(warm + n_batches):
        seeds = torch.from_numpy(seed_rs.randint(0, N_NODES, size=per_step).astype(np.int32))
        t0 = time.perf_counter()
        torch_ref.forward(adj_t, feats_t, seeds, FANOUT, aggs, concat, kind, 123, 2 * i, normalize=True)
        dt = time.perf_counter() - t0
        if i >= warm:
            times.append(dt)
    return per_step * len(times) / sum(times), torch.get_num_threads(), float(np.median(times))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=500)
    ap.add_argument("--warmup", type=int, default=30)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--aggregator", default="mean", choices=["mean", "gcn", "maxpool"],
                    help="mean = BASELINE configs[1] (default); maxpool (+ bf16 features, --math bf16) = configs[2]")
    ap.add_argument("--math", default=os.environ.get("GS_MATH", "tf32x3"),
                    help="tf32x3 (tcgen05, fp32-grade: meets the 1e-4 parity bar) | fp32 (CUDA cores) | tf32 | bf16")
    ap.add_argument("--cpu-batches", type=int, default=12)
    ap.add_argument("--depth", type=int, default=int(os.environ.get("GS_PIPE_DEPTH", "4")),
                    help="graph runners / compute streams alternating in the pipelined front end")
    ap.add_argument("--no-partitioned", action="store_true", help="skip the node-partitioned measurement at N > 1")
    ap.add_argument("--repeats", type=int, default=1,
                    help="how many times each K-step timed region is repeated (median reported); 0 = auto (~0.3 s per leg)")
    ap.add_argument("--no-config3", action="store_true", help="skip the short max-pool/bf16 pass behind roofline_tensor")
    ap.add_argument("--workload", default="reddit", choices=["reddit", "unsup", "rmat", "train"],
                    help="reddit = BASELINE configs[1] (default; the contract line); unsup = configs[3]: unsupervised training "
                         "step, node-partitioned, data parallel; rmat = configs[4]: R-MAT graph, CSR sampler, partitioned")
    ap.add_argument("--rmat-scale", type=int, default=20, help="log2 of the R-MAT id space (27 = BASELINE configs[4])")
    ap.add_argument("--rmat-nodes", type=int, default=0, help="nodes after trimming (0 = 2^scale; 100000000 for configs[4])")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the last step's output embeddings to DIR/embeddings.npy")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "ours" or args.workload != "reddit"):
        ap.error("--dump-outputs covers the CUDA path of the reddit workload")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    kind = args.aggregator
    if kind == "maxpool":
        args.math = "bf16"            # config 3: bf16 features / weights, fp32 accumulate, K4 on tcgen05
    workload = "reddit-shape synthetic N=%d F=%d max_degree=%d graphsage_%s 2-hop fanout 25x10 batch=%d dims=[%d,%d,%d]" % (
        N_NODES, F, MAX_DEG, kind, BATCH, F, DIM, DIM)

    # ------------------------------------------------------------------ reference arm (CPU)
    if args.impl == "reference":
        if rank != 0:
            return
        g = build_graph()
        w = make_weights(kind, np.random.RandomState(7))
        t0 = time.perf_counter()
        rate, cores, med = cpu_reference_rate(g, kind, w, args.steps, args.warmup, np.random.RandomState(1000),
                                              budget_s=150.0)
        per_step = cpu_reference_rate.per_step
        print(json.dumps({
            "impl": "reference", "metric": "seed_nodes_per_sec", "value": rate, "unit": "nodes/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": med * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": bench_config(workload, kind),
            "impl_detail": {"note": "reference op sequence restated on torch-CPU (TensorFlow 1.x unavailable offline)"},
            "cpu_baseline": {"value": rate, "unit": "nodes/s", "cores": cores, "kind": "port",
                             "sample": "%d steps of %d seeds each (fanout 25x10, same graph/weights)" % (args.steps, per_step)},
            "e2e": {"value": rate, "unit": "nodes/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}))
        return

    # ------------------------------------------------------------------ our arm (B200)
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    import graphsage_b200 as gs
    from graphsage_b200 import ops

    dev = torch.device("cuda", local_rank)
    if args.workload == "rmat":
        import bench_extra
        return bench_extra.run_rmat(args, rank, world, local_rank, dist, dev)
    g = build_graph(rank, world, (lambda: dist.barrier()) if dist is not None else None)
    if args.workload == "unsup":
        import bench_extra
        return bench_extra.run_unsup(args, g, rank, world, local_rank, dist, dev)
    if args.workload == "train":
        import bench_extra
        return bench_extra.run_train(args, g, rank, world, local_rank, dist, dev)
    tdtype = torch.bfloat16 if kind == "maxpool" else torch.float32
    table = torch.zeros((N_NODES + 1, ops.pad_cols(F)), dtype=tdtype, device=dev)
    table[:, :F] = torch.from_numpy(g["features"]).to(dev).to(tdtype)
    adj_dev = torch.from_numpy(g["adj"]).to(dev)
    gs.set_default_math(args.math)
    sampler = gs.UniformNeighborSampler(adj_dev, seed=123)
    dims = (2 * DIM, 2 * DIM) if kind == "gcn" else (DIM, DIM)
    infos = [gs.SAGEInfo("node", sampler, FANOUT[0], dims[0]), gs.SAGEInfo("node", sampler, FANOUT[1], dims[1])]
    model = gs.SampleAndAggregate({"batch_size": BATCH, "dropout": 0.}, table[:, :F], adj_dev, None, infos,
                                  concat=(kind != "gcn"), aggregator_type=kind, device=dev)
    weights = make_weights(kind, np.random.RandomState(7))
    weights_by_kind = {kind: weights}

    def weights_for(mdl):
        k_ = getattr(mdl, "_bench_kind", kind)
        if k_ not in weights_by_kind:
            weights_by_kind[k_] = make_weights(k_, np.random.RandomState(7))
        return weights_by_kind[k_]

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if dist is None:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    R = args.repeats if args.repeats > 0 else int(min(200, max(5, np.ceil(4000.0 / max(args.steps, 1)))))
    total = args.warmup + args.steps * R

    def stats(ms_list):
        a = np.sort(np.asarray(ms_list, dtype=np.float64))
        return {"median": float(np.median(a)), "p10": float(a[int(0.1 * (len(a) - 1))]), "p90": float(a[int(np.ceil(0.9 * (len(a) - 1)))]),
                "min": float(a[0]), "max": float(a[-1]), "n": int(len(a))}

    def measure(mdl, lo, hi, tag, probe_name, do_e2e=True, reps=R):
        """value (ids resident in HBM) and e2e (pinned-host ids in, result to pinned host) for one model.  Each timed
        region is EXACTLY args.steps steps; it is repeated `reps` times back to back (fresh seeds every step) and the
        median region is reported, so a 20-step / 1.6 ms region no longer rides on one PCIe or scheduling hiccup."""
        rs = np.random.RandomState(1000 + rank)
        n_total = args.warmup + args.steps * reps
        seeds_host = torch.from_numpy(rs.randint(lo, hi, size=(n_total, BATCH)).astype(np.int32)).pin_memory()
        seeds_dev = seeds_host.to(dev)
        out_host = torch.empty((args.steps, BATCH, 2 * DIM), dtype=torch.float32).pin_memory()
        mdl.forward(seeds_dev[0])                       # creates the aggregators
        for a, w in zip(mdl.aggregators, weights_for(mdl)):
            for k_, v in w.items():
                if k_ == "mlp_weights":
                    a.mlp_layers[0].vars["weights"] = torch.from_numpy(v).to(dev)
                elif k_ == "mlp_bias":
                    a.mlp_layers[0].vars["bias"] = torch.from_numpy(v).to(dev)
                else:
                    a.vars[k_] = torch.from_numpy(v).to(dev)
        # ---- timed region 1 ("value"): ids resident in HBM, one CUDA graph per step; `depth` runners alternate on their
        #      own streams (steps are independent), so one step's sampler + gather overlaps the previous step's GEMMs
        pipe = mdl.pipelined(BATCH, normalize=True, depth=args.depth)
        cur = torch.cuda.current_stream(dev)
        clocks = ClockSampler(local_rank)      # NVML start-up perturbs the steps around it: keep it in the warm-up
        clocks.start()
        for i in range(args.warmup):
            pipe.submit_device(seeds_dev[i])
        pipe.synchronize()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ms_value = []
        for rep in range(reps):
            base = args.warmup + rep * args.steps
            for c in pipe.computes:
                c.wait_stream(cur)
            e0.record(cur)
            for c in pipe.computes:
                c.wait_event(e0)
            for i in range(args.steps):
                out = pipe.submit_device(seeds_dev[base + i])
            for c in pipe.computes:
                cur.wait_stream(c)
            e1.record(cur)
            pipe.synchronize()
            barrier()
            ms_value.append(max_over_ranks(e0.elapsed_time(e1)))
        last_output = out.float().cpu().numpy() if args.dump_outputs else None   # the last timed step's result
        clk = clocks.summary()
        launches_per_step = pipe.runners[0].launches_per_replay
        pipe.close()
        # ---- timed region 2 (roofline): same steps with the dominant kernel isolated in its own graph node and
        #      bracketed by CUDA events on the launching stream (the split costs two extra graph launches per step)
        runner = mdl.graphed(BATCH, normalize=True, probe=probe_name)
        for i in range(min(args.warmup, 5)):
            runner(seeds_dev[i])
        barrier()
        n_probe = args.steps * min(reps, 5)
        pev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(n_probe)]
        e0.record()
        for i in range(n_probe):
            runner(seeds_dev[args.warmup + i], probe_events=pev[i])
        e1.record()
        barrier()
        ms_probe_total = max_over_ranks(e0.elapsed_time(e1))
        runner.close()
        kernel_ms = float(np.mean([a.elapsed_time(b) for a, b in pev]))
        res = dict(ms_value=stats(ms_value), clocks=clk, launches=launches_per_step * args.steps,
                   launches_per_step=launches_per_step, ms_probe_step=ms_probe_total / n_probe,
                   gather_kernel_ms=max_over_ranks(kernel_ms), reps=reps, last_output=last_output)
        res["ms_total"] = res["ms_value"]["median"]
        res["value"] = world * BATCH * args.steps / (res["ms_total"] * 1e-3)
        if not do_e2e:
            return res
        # end to end through the public host-buffer API: pinned ids in, result in pinned host memory, every step
        pipe = mdl.pipelined(BATCH, normalize=True, depth=args.depth)
        for i in range(min(args.warmup, 6)):
            pipe.submit(seeds_host[i], out_host[i % args.steps])
        pipe.synchronize()
        barrier()
        ms_e2e = []
        for rep in range(reps):
            base = args.warmup + rep * args.steps
            e0.record(pipe.compute)
            for i in range(args.steps):
                pipe.submit(seeds_host[base + i], out_host[i])
            pipe.copy.wait_stream(pipe.compute)
            e1.record(pipe.copy)                                # after the last result has reached the host buffer
            pipe.synchronize()
            barrier()
            ms_e2e.append(max_over_ranks(e0.elapsed_time(e1)))
        pipe.close()
        chk = float(out_host[-1].abs().sum())                  # the host really received the last result
        assert np.isfinite(chk) and chk > 0
        res["ms_e2e_stats"] = stats(ms_e2e)
        res["ms_e2e"] = res["ms_e2e_stats"]["median"]
        res["e2e"] = world * BATCH * args.steps / (res["ms_e2e"] * 1e-3)
        return res

    def probe_of(k_):
        return ("maxpool_mlp/%d" % (BATCH * 10)) if k_ == "maxpool" else ("gather_mean/%d" % (BATCH * 11))

    def build_model(k_, feats_table, math):
        gs.set_default_math(math)
        smp = gs.UniformNeighborSampler(adj_dev, seed=123)
        d_ = (2 * DIM, 2 * DIM) if k_ == "gcn" else (DIM, DIM)
        inf = [gs.SAGEInfo("node", smp, FANOUT[0], d_[0]), gs.SAGEInfo("node", smp, FANOUT[1], d_[1])]
        mdl = gs.SampleAndAggregate({"batch_size": BATCH, "dropout": 0.}, feats_table, adj_dev, None, inf,
                                    concat=(k_ != "gcn"), aggregator_type=k_, device=dev)
        mdl._bench_kind = k_
        return mdl, inf

    def hbm_roofline(res):
        peak, peak_src = peaks()
        avg_ms = res["gather_kernel_ms"]
        achieved = GATHER_BYTES / (avg_ms * 1e-3) / 1e9
        traffic, src = None, None           # dram__bytes_read + dram__bytes_write of this kernel, committed ncu capture
        for name in ("ncu_gather_r02_summary.txt", "ncu_gather_r01_final_summary.txt"):
            prof = os.path.join(ROOT, "profiles", name)
            if not os.path.exists(prof):
                continue
            vals = {}
            for line in open(prof):
                if line.strip() == "" and vals:
                    break                                    # first kernel record = the layer-0 launch
                if line.startswith("dram__bytes_") and "=" in line:
                    k_, v_ = line.split("=")
                    vals[k_.strip()] = float(v_.split()[0]) * 1e6
            if len(vals) == 2:
                traffic, src = sum(vals.values()), "profiles/%s (ncu --set full, one launch; bytes)" % name
                break
        step_ms = res["ms_total"] / args.steps
        return {"bound": "hbm", "kernel": "gather_mean (layer 0, hops 0+1: fused 2-hop feature gather + fanout mean)",
                "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                "traffic_source": src, "peak_source": peak_src, "avg_kernel_ms": avg_ms,
                "algorithmic_bytes_per_launch": GATHER_BYTES,
                "kernel_share_of_step": avg_ms / step_ms,
                "kernel_share_of_probed_step": avg_ms / res["ms_probe_step"],
                "step_hbm_frac": (GATHER_BYTES + 2.5e6) / (step_ms * 1e-3) / 1e9 / peak,
                "measured_in": "second timed pass of the same steps with this kernel isolated in its own CUDA-graph node "
                               "(%.1f us/step there, serial); kernel_share_of_step divides by the headline pipelined step "
                               "(%.1f us), where kernels of neighbouring steps overlap" % (res["ms_probe_step"] * 1e3, step_ms * 1e3)}

    def tensor_roofline(res):
        avg_ms = res["gather_kernel_ms"]
        flops = 2.0 * BATCH * 250 * F * 512                       # hop-2 MLP: [128000, 602] x [602, 512]
        tpeak, tburst = 1444.6, 1725.0
        pk = os.path.join(ROOT, "MEASURED_PEAKS.json")
        if os.path.exists(pk):
            d_ = json.load(open(pk))
            tpeak, tburst = float(d_.get("bf16_tflops_sustained", tpeak)), float(d_.get("bf16_tflops", tburst))
        ach = flops / (avg_ms * 1e-3) / 1e12
        traffic, src = None, None
        prof = os.path.join(ROOT, "profiles", "ncu_maxpool_r02_summary.txt")
        if os.path.exists(prof):
            vals = {}
            for line in open(prof):
                if line.startswith("dram__bytes_") and "=" in line and len(vals) < 2:
                    k_, v_ = line.split("=")
                    vals[k_.strip()] = float(v_.split()[0]) * 1e6
            if len(vals) == 2:
                traffic, src = sum(vals.values()), "profiles/ncu_maxpool_r02_summary.txt"
        return {"bound": "tensor", "kernel": "maxpool_mlp (layer 0, hop 2: gather + MLP 602->512 + ReLU + max over 25), tcgen05 bf16",
                "achieved": ach, "peak": tpeak, "unit": "TFLOP/s", "frac": ach / tpeak, "frac_of_burst_peak": ach / tburst,
                "traffic": traffic, "traffic_source": src,
                "peak_source": "measured sustained cuBLAS bf16 (MEASURED_PEAKS.json); burst %.0f" % tburst,
                "avg_kernel_ms": avg_ms, "algorithmic_flops_per_launch": flops,
                "kernel_share_of_step": avg_ms / (res["ms_total"] / args.steps),
                "kernel_share_of_probed_step": avg_ms / res["ms_probe_step"]}

    # replicated table: every rank holds the 561 MB table and runs its own seed batches (no data-path collective)
    model._bench_kind = kind
    rep = measure(model, 0, N_NODES, "replicated", probe_of(kind))

    # node-partitioned table with the halo exchange fused into the gather (peer loads over NVLink); owner-computes seeds
    part = None
    if world > 1 and not args.no_partitioned and kind != "maxpool":
        from graphsage_b200 import parallel
        bounds = parallel.community_bounds(g["comm"], world)      # cuts moved to community starts: no community straddles
        lo, hi = bounds[rank], bounds[rank + 1]
        def run_partitioned(cache_rows, full):
            hot = parallel.hot_remote_rows(g["adj"], N_NODES, world, rank, cache_rows, row_start=bounds)
            shard = parallel.ShardedFeatures(g["features"][lo:hi], N_NODES, row_start=bounds, replica_ids=hot,
                                             replica_rows=g["features"][hot])
            model_p, infos_p = build_model(kind, shard, args.math)
            pr = measure(model_p, lo, hi, "partitioned", probe_of(kind), do_e2e=full, reps=R if full else max(1, min(R, 5)))
            rs = np.random.RandomState(1000 + rank)
            smp, _ = model_p.sample(torch.from_numpy(rs.randint(lo, hi, size=BATCH).astype(np.int32)).to(dev), infos_p)
            allids = torch.cat(smp)
            rho_part = max_over_ranks(shard.remote_fraction(allids, use_replicas=False))
            rho = max_over_ranks(shard.remote_fraction(allids))
            out = {"value": pr["value"], "unit": "nodes/s", "ms_per_step": pr["ms_total"] / args.steps,
                   "remote_row_fraction_by_partition": rho_part, "remote_row_fraction_after_replicas": rho,
                   "replica_rows_per_gpu": int(len(hot)), "replica_fraction_of_table": float(len(hot)) / N_NODES,
                   "gather_kernel_ms": pr["gather_kernel_ms"],
                   "nvlink_GBps_per_gpu": rho * GATHER_BYTES / (pr["gather_kernel_ms"] * 1e-3) / 1e9,
                   "nvlink_peak_GBps": 770.0, "halo_staging": bool(shard.stage_halo)}
            if shard.stage_halo:
                # with staging the gather kernel reads local memory only; the NVLink transfer is the fetch pass, which
                # overlaps the neighbouring steps - its rate is bounded below by (unique remote bytes / step time)
                uniq = float(torch.unique(allids[(parallel.owner_of(allids, N_NODES, world, bounds) != rank) & (allids < N_NODES)
                                                  & ((shard.remap[allids.clamp(0, N_NODES).long()] < 0) if shard.remap is not None else True)]).numel())
                out["unique_remote_rows_per_step"] = uniq
                out["nvlink_GBps_per_gpu"] = uniq * F * 4 / (out["ms_per_step"] * 1e-3) / 1e9
                out["nvlink_note"] = "unique remote rows of one step x row bytes / pipelined step time (lower bound on the fetch pass's rate)"
            if full:
                out.update({"e2e": pr["e2e"], "e2e_ms_per_step": pr["ms_e2e"] / args.steps, "value_spread_ms": pr["ms_value"],
                            "last_output": pr["last_output"],
                            "clocks": pr["clocks"], "launches": pr["launches"],
                            "partition": "community-aligned contiguous ranges, %d..%d rows per GPU" % (
                                min(np.diff(bounds)), max(np.diff(bounds))),
                            "note": "node-partitioned features (contiguous community-aligned ranges), adjacency replicated, "
                                    "remote rows pulled by the gather kernel over NVLink peer mappings (one bulk copy per row), "
                                    "the hottest remote rows replicated locally (budget: 1/4 of the table per GPU unless "
                                    "GS_HALO_CACHE_ROWS says otherwise), (GS_HALO_STAGING=1 adds the opt-in halo staging passes); owner-computes seeds"})
            barrier()
            shard.close()
            return out

        cache_rows = int(os.environ.get("GS_HALO_CACHE_ROWS", str(parallel.default_cache_rows(N_NODES, world))))
        part = run_partitioned(cache_rows, True)
        sweep = os.environ.get("GS_HALO_CACHE_SWEEP", "")
        if sweep:
            part["replica_sweep"] = [run_partitioned(int(float(f) * N_NODES), False) for f in sweep.split(",") if f.strip()]

    # config 3 (BASELINE configs[2]) in the same run: max-pool aggregator over a bf16 table, K4 on tcgen05
    c3 = None
    if kind == "mean" and world == 1 and not args.no_config3:
        table3 = torch.zeros((N_NODES + 1, ops.pad_cols(F)), dtype=torch.bfloat16, device=dev)
        table3[:, :F] = table[:, :F].to(torch.bfloat16)
        model3, _ = build_model("maxpool", table3[:, :F], "bf16")
        c3 = measure(model3, 0, N_NODES, "config3", probe_of("maxpool"), do_e2e=False, reps=max(1, min(R, 5)))
        gs.set_default_math(args.math)

    if rank != 0:
        return
    head = part if part is not None else None
    last_output = (head if head is not None else rep).pop("last_output")
    if args.dump_outputs:
        os.makedirs(args.dump_outputs, exist_ok=True)
        np.save(os.path.join(args.dump_outputs, "embeddings.npy"), last_output)
    roof = (tensor_roofline(rep) if kind == "maxpool" else hbm_roofline(rep)) if rep["gather_kernel_ms"] > 0 else None
    cpu = None
    if world == 1 and args.cpu_batches > 0:
        rate, cores, med = cpu_reference_rate(g, kind, weights, args.cpu_batches, 2, np.random.RandomState(1000))
        cpu = {"value": rate, "unit": "nodes/s", "cores": cores, "kind": "port",
               "sample": "%d batches of %d seeds, same graph/weights, torch-CPU restatement of the reference op sequence"
                         % (args.cpu_batches, BATCH), "ms_per_batch_median": med * 1e3}
    line = {
        "metric": "seed_nodes_per_sec", "value": rep["value"], "unit": "nodes/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": rep["ms_total"] / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "bf16" if kind == "maxpool" else "f32", "data": "synthetic",
        "config": bench_config(workload, kind),
        "impl_detail": {"math": args.math, "pipeline_depth": args.depth,
                        "parallelism": "replicated-table dp%d" % world,
                        "timing": "each K-step region repeated %d times back to back, median reported" % rep["reps"]},
        "e2e": {"value": rep["e2e"], "unit": "nodes/s", "h2d_bytes_per_step": BATCH * 4,
                "d2h_bytes_per_step": BATCH * 2 * DIM * 4, "ms_per_step": rep["ms_e2e"] / args.steps,
                "region_ms": rep["ms_e2e_stats"]},
        "value_region_ms": rep["ms_value"],
        "gpu_launches": rep["launches"], "clocks": rep["clocks"], "roofline": roof, "cpu_baseline": cpu,
        "kernel_ms": {probe_of(kind): rep["gather_kernel_ms"]}, "partitioned": part}
    if head is not None:
        # N > 1: the headline is the node-partitioned engine north_star asks for; the replicated-table numbers stay
        # beside it (they need no exchange at all, so they say nothing about the halo path)
        line["replicated"] = {"value": rep["value"], "ms_per_step": rep["ms_total"] / args.steps, "e2e": rep["e2e"],
                              "note": "every rank holds the whole 561 MB table; no data-path exchange"}
        line.update({"value": head["value"], "ms_per_step": head["ms_per_step"], "gpu_launches": head["launches"],
                     "clocks": head["clocks"], "value_region_ms": head["value_spread_ms"]})
        line["e2e"] = {"value": head["e2e"], "unit": "nodes/s", "h2d_bytes_per_step": BATCH * 4,
                       "d2h_bytes_per_step": BATCH * 2 * DIM * 4, "ms_per_step": head["e2e_ms_per_step"]}
        line["impl_detail"]["parallelism"] = "node-partitioned x%d, halo rows over NVLink peer mappings" % world
    if c3 is not None:
        line["roofline_tensor"] = tensor_roofline(c3)
        line["config3"] = {"workload": "same graph, graphsage_maxpool bf16 (BASELINE configs[2])", "value": c3["value"],
                           "unit": "nodes/s", "ms_per_step": c3["ms_total"] / args.steps, "region_ms": c3["ms_value"],
                           "gpu_launches": c3["launches"], "launches_per_step": c3["launches_per_step"]}
    print(json.dumps(line))


if __name__ == "__main__":
    try:
        main()
    finally:
        import torch.distributed as _dist
        if _dist.is_available() and _dist.is_initialized():
            _dist.destroy_process_group()
