#!/usr/bin/env python
"""Benchmark of the hot path: batched VE posterior queries (headline) + CPT-fit counting, all five BASELINE.json configs.

    python bench.py --gpus N --steps K --warmup W            # our arm (one process per GPU under torchrun)
    python bench.py --impl reference --steps K --warmup W    # the reference-style CPU path (oracle port) on the host cores
    python bench.py --steps K --warmup W --dump-outputs bench_outputs   # also write the headline's posteriors (seeded row sample)

Headline workload = BASELINE.json configs[2], the configuration the metric's "at 1/2/4/8 B200" is quoted on: Alarm-shaped
network (37 nodes, card <= 4), 16,777,216 evidence rows in total, row-sharded over the ranks (STRONG scaling), evidence =
12 observable leaves drawn from the joint, targets HYPOVOLEMIA / LVFAILURE / KINKEDTUBE / PULMEMBOLUS answered by one fused
launch.  One *pass* = the fused plan over the rank's shard of one 16M-row batch; one *query* = one posterior row of one
target.  One *step* = P consecutive passes, P chosen (and reported) so that the K timed steps cover >= 60 ms of device time:
a single pass is 20-160 microseconds, far too short to time alone.  The K steps are CUDA-graph replays (one graph = one
step), bracketed by barrier + synchronize, timed with CUDA events on the launch stream, MAX over ranks.
Inputs are device resident for `value`; a batch (evidence + posteriors) is larger than L2, or the passes rotate through a
ring of distinct batches that is (stated in `config.l2`).  `e2e` runs the same workload through the C-ABI host-buffer call
(pinned host codes in, pinned host posteriors out, copies inside the timed region); `e2e.python_api` is the reference-facing
`infer(target, {name: float32 [nq,1]})`.

Every configuration also gets its own object (`configs.<name>`) with value / roofline / cpu_baseline / e2e where they
apply; compact copies sit inside the top-level `roofline`, `cpu_baseline` and `e2e` objects (`per_config`).
Prints ONE JSON line on rank 0.
"""
import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

ASIA_EVIDENCE = ["asia", "smoke", "xray", "dysp"]
ASIA_TARGETS = ["lung", "tub", "bronc"]
ALARM_ROWS = 1 << 24
L2_BYTES = 126 * 1024 * 1024
METRIC = "posterior queries/sec (batched VE)"
MIN_REGION_S = 0.060
# --dump-outputs: 3 batches x 4 targets x 2^18 rows x 2 fp32 = 24 MiB of posteriors (the ring always holds >= 3 batches)
DUMP_ROWS, DUMP_BATCHES, DUMP_SEED = 1 << 18, 3, 1250
# identical in both arms (the driver compares them): what is computed, not how
CONFIG = {"workload": "alarm-37node batched VE (BASELINE.json configs[2]): 16,777,216 evidence rows in total, 12 evidence "
                      "leaves drawn from the joint, 4 binary targets (HYPOVOLEMIA, LVFAILURE, KINKEDTUBE, PULMEMBOLUS)",
          "rows_total": ALARM_ROWS, "targets": 4, "queries_per_pass": ALARM_ROWS * 4,
          "cpts": "fitted from forward samples of seeded Dirichlet CPTs on the published Alarm structure",
          "step": "one step = P consecutive passes over 16M-row batches, P chosen so that the K timed steps cover >= 60 ms of device "
                  "time (run_detail.passes_per_step); the CPU arm's step is a bounded sample of one pass (cpu_baseline.sample)",
          "l2": "GPU arm: the passes rotate through a ring of >= 3 distinct resident batches (evidence codes + posteriors, 738 MB / n_gpus "
                "each per GPU) that together exceed 2 x the 126 MB L2 (run_detail.l2); inputs resident in HBM for `value`, in pinned "
                "host memory for `e2e`"}


def _peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def _profile_traffic(kernel_key):
    """dram bytes per launch of a kernel from the committed ncu summary (profiles/traffic.json), or None."""
    try:
        return json.load(open(os.path.join(ROOT, "profiles", "traffic.json"))).get(kernel_key)
    except Exception:
        return None


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""

    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.lines, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "20"], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.05)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for l in self.lines:
            parts = [x.strip() for x in l.split(",")]
            if len(parts) < 6:
                continue
            try:
                sm.append(float(parts[0])); mx = float(parts[1])
            except ValueError:
                continue
            for nm, v in zip(names, parts[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


# ================================================================================================ CPU legs (oracle)
def _cpu_threads():
    import torch

    torch.set_num_threads(os.cpu_count() or 1)
    return torch.get_num_threads()


def _oracle_net_from_samples(spec, n_fit, seed):
    """CPTs fitted by the oracle from forward samples (numpy restatement of the sampler): the CPU arm's network."""
    from continuousbayesiannetwork_b200 import synth
    from oracle import cbn_oracle as O

    codes = synth.sample_forward_numpy(spec, seed, 0, n_fit)
    fitted = [O.cpt_from_counts(O.dense_counts(codes, spec.parents[i] + [i], spec.cards), n_fit)[1] for i in range(spec.n)]
    return O.DiscreteNet(spec.cards, spec.parents, fitted)


def cpu_ve(spec, net, evidence, targets, rows_per_call, budget_s, seed=11, label=""):
    """oracle O2 (textbook batched VE, fp32 PyTorch on all host cores) on a bounded sample of a query workload."""
    from continuousbayesiannetwork_b200 import synth
    from oracle import cbn_oracle as O

    cores = _cpu_threads()
    ids = [spec.names.index(e) for e in evidence]
    ev = synth.sample_forward_numpy(spec, seed, 0, rows_per_call)[ids].T
    O.ve_posterior(net, spec.names.index(targets[0]), ids, ev[:256])           # warm-up
    done, calls, t0 = 0, 0, time.perf_counter()
    while True:
        for t in targets:
            O.ve_posterior(net, spec.names.index(t), ids, ev)
        done += rows_per_call * len(targets)
        calls += 1
        el = time.perf_counter() - t0
        if el >= budget_s:
            break
    return {"value": done / el, "unit": "queries/s", "cores": cores, "kind": "port",
            "sample": f"{done} queries = {calls} x ({rows_per_call} rows x {len(targets)} targets) of the {label} workload in {el:.1f}s; "
                      "oracle O2 = textbook batched VE in fp32 PyTorch (the reference has no correct multi-layer query path, SURVEY.md 3.3)"}


def cpu_fit(spec, n, budget_s, seed=5, label=""):
    """The reference's fit arithmetic (BruteForce._fit, brute_force.py:17-53: torch.unique(dim=0) sort + counts, restated as
    oracle.fit_mle) per node on n forward samples, all host cores; nodes are timed until the budget is used and the
    whole-network rate is n / (mean node time x number of nodes)."""
    import torch

    from continuousbayesiannetwork_b200 import synth
    from oracle import cbn_oracle as O

    cores = _cpu_threads()
    codes = synth.sample_forward_numpy(spec, seed, 0, n)
    cols = [torch.from_numpy(codes[i].astype("float32")) for i in range(spec.n)]
    order = sorted(range(spec.n), key=lambda i: -len(spec.parents[i]))
    order = order[:: max(1, len(order) // 16)] if spec.n > 40 else list(range(spec.n))     # a 16-node spread for big networks
    times, t_all = [], time.perf_counter()
    for i in order:
        pa = torch.stack([cols[p] for p in spec.parents[i]]) if spec.parents[i] else None
        t0 = time.perf_counter()
        O.fit_mle(cols[i], pa)
        times.append(time.perf_counter() - t0)
        if time.perf_counter() - t_all > budget_s:
            break
    per_node = sum(times) / len(times)
    return {"value": n / (per_node * spec.n), "unit": "samples/s", "cores": cores, "kind": "port",
            "sample": f"oracle.fit_mle (torch.unique sort path of BruteForce._fit) on n={n} samples, {len(times)} of {spec.n} nodes of "
                      f"{label} timed ({sum(times):.1f}s), extrapolated to the whole network"}


def run_reference(args):
    """The reference's CPU implementation of the headline path: oracle O2 on all host cores, same config / metric / unit;
    each step is a bounded sample of the 16M-row pass."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from continuousbayesiannetwork_b200 import synth
    from oracle import cbn_oracle as O

    cores = _cpu_threads()
    spec = synth.alarm()
    net = _oracle_net_from_samples(spec, 200_000, 1236)
    rows = args.ref_rows
    ids = [spec.names.index(e) for e in synth.ALARM_EVIDENCE]
    ev = synth.sample_forward_numpy(spec, 11, 0, rows)[ids].T

    def step():
        for t in synth.ALARM_TARGETS:
            O.ve_posterior(net, spec.names.index(t), ids, ev)

    for _ in range(args.warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step()
    el = time.perf_counter() - t0
    val = rows * len(synth.ALARM_TARGETS) * args.steps / el
    sample = (f"each step = {rows} evidence rows x 4 targets, a bounded sample of the 16,777,216-row pass; oracle O2 = textbook "
              "batched VE in fp32 PyTorch on the host cores (reference-style PyTorch path: the reference has no correct "
              "multi-layer query routine, SURVEY.md 3.3); CPTs fitted by the oracle from 200,000 forward samples")
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": "queries/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": el / args.steps * 1e3, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": CONFIG,
            "cpu_baseline": {"value": val, "unit": "queries/s", "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": val, "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


def _bind_to_gpu_numa_node(index):
    """One process per GPU: run (and first-touch the pinned staging memory) on the CPU cores next to that GPU, so the
    host<->device copies of the e2e path do not cross the socket interconnect.  Returns (cpus before, cpus after)."""
    before = after = None
    try:
        import pynvml

        before = os.sched_getaffinity(0)
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        n_cpu = os.cpu_count() or 1
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (n_cpu + 63) // 64)
        cpus = [w * 64 + b for w, m in enumerate(words) for b in range(64) if (m >> b) & 1 and w * 64 + b < n_cpu]
        allowed = sorted(set(cpus) & set(before))
        if allowed:
            os.sched_setaffinity(0, allowed)
        after = os.sched_getaffinity(0)
    except Exception:
        pass
    return before, after


# ================================================================================================ our arm
class Env:
    def __init__(self):
        import torch
        import torch.distributed as dist

        self.torch, self.dist = torch, dist
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        torch.cuda.set_device(self.local)
        self.dev = torch.device("cuda", self.local)
        self.cpus_before, self.cpus_bound = _bind_to_gpu_numa_node(self.local)
        if self.world > 1:
            dist.init_process_group("nccl", device_id=self.dev)
        self.peak, self.peak_src = _peaks()

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, x):
        if self.world == 1:
            return float(x)
        t = self.torch.tensor([x], dtype=self.torch.float64, device=self.dev)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def timed(self, fn, steps, warmup):
        """W untimed calls, then exactly K calls bracketed by barrier + synchronize; CUDA events on the launch stream;
        MAX over ranks.  Returns seconds."""
        torch = self.torch
        for i in range(warmup):
            fn(i)
        self.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(steps):
            fn(warmup + i)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        self.barrier()
        return self.max_over_ranks(ms) / 1e3

    def host_timed(self, fn, steps, warmup):
        """Host clock around synchronous calls (each returns after its last D2H copy has landed)."""
        for i in range(warmup):
            fn(i)
        self.barrier()
        t0 = time.perf_counter()
        for i in range(steps):
            fn(warmup + i)
        self.torch.cuda.synchronize()
        el = time.perf_counter() - t0
        self.barrier()
        return self.max_over_ranks(el)

    def graph_of(self, passes, streams=1):
        """ONE CUDA graph holding the given launch closures in order; with streams > 1 consecutive (independent) passes are
        spread round-robin over that many streams inside the graph (what a serving loop does)."""
        torch = self.torch
        side = [torch.cuda.Stream(device=self.dev) for _ in range(streams - 1)]
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            main = torch.cuda.current_stream()
            for s in side:
                s.wait_stream(main)
            for i, p in enumerate(passes):
                k = i % streams
                if k == 0:
                    p()
                else:
                    with torch.cuda.stream(side[k - 1]):
                        p()
            for s in side:
                main.wait_stream(s)
        return g

    def passes_per_step(self, one_pass, steps, ring, min_region_s=MIN_REGION_S):
        """P such that `steps` steps of P passes cover >= min_region_s (agreed over the ranks; a multiple of the ring)."""
        torch = self.torch
        for i in range(3):
            one_pass(i)
        self.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(10):
            one_pass(i)
        e1.record()
        torch.cuda.synchronize()
        est = self.max_over_ranks(e0.elapsed_time(e1) / 1e3 / 10)
        margin = 1.15
        if est < 50e-6:
            margin = 1.5          # the long graph of the timed region overlaps consecutive launches better than this short one
            # launch-latency scale: eager launches overestimate the pass; time a small graph of passes instead
            n = max(ring, 8) * 4
            g = self.graph_of([(lambda j=j: one_pass(j)) for j in range(n)])
            g.replay()
            self.barrier()
            e0.record()
            g.replay()
            e1.record()
            torch.cuda.synchronize()
            est = min(est, self.max_over_ranks(e0.elapsed_time(e1) / 1e3 / n))
            del g
        p = max(1, math.ceil(margin * min_region_s / (steps * est)))
        p = min(p, 4096)
        return (p + ring - 1) // ring * ring, est


def roofline(env, alg_bytes_per_launch, launch_s, kernel, traffic_key=None, extra=None):
    ach = alg_bytes_per_launch / launch_s / 1e9
    r = {"bound": "hbm", "achieved": ach, "peak": env.peak, "unit": "GB/s", "frac": ach / env.peak,
         "traffic": _profile_traffic(traffic_key or kernel), "kernel": kernel,
         "algorithmic_bytes_per_launch": alg_bytes_per_launch, "launch_us": launch_s * 1e6, "peak_source": env.peak_src}
    if extra:
        r.update(extra)
    return r


def verify_sharded_fit(env, spec, tables, seed, n_per_rank):
    """After a sharded fit: rank 0 recounts the CONCATENATED shards alone (no collective) and requires bit-equal tables
    and sample count.  Returns a short status string (asserts on mismatch)."""
    torch = env.torch
    from continuousbayesiannetwork_b200.engine import sample_network, tables_from_spec

    ok = True
    if env.rank == 0:
        alone = tables_from_spec(spec, env.dev)
        buf = None
        for r in range(env.world):
            buf = sample_network(spec, seed=seed, first=r * n_per_rank, n=n_per_rank, device=env.dev, tables=alone, out=buf)
            alone.count(buf, n_per_rank)
        ok = bool(torch.equal(alone.counts, tables.counts)) and alone.n_total == tables.n_total
        del alone, buf
    env.barrier()
    assert ok, "all-reduced count tables differ from the single-GPU recount of the concatenated shards"
    return f"rank 0 recounted the {env.world} concatenated shards alone: tables and n_total bit-equal"


def dump_headline_outputs(env, out_dir, out_ring, targets, first_row):
    """--dump-outputs: the posteriors the last timed step of the headline left in the first DUMP_BATCHES batches of the ring
    (every step covers the whole ring), at DUMP_ROWS rows drawn with a fixed seed from the 16M-row batch.  Row ids are global,
    so the files do not depend on the number of GPUs.  Writes `<target>_batch<r>.npy` (float32 [DUMP_ROWS, card]) and
    `rows.npy` (the sampled row ids, float64) on rank 0."""
    import numpy as np

    torch = env.torch
    idx = np.sort(np.random.default_rng(DUMP_SEED).choice(ALARM_ROWS, size=DUMP_ROWS, replace=False))
    n_local = out_ring[0][0].shape[0]
    mine = (idx >= first_row) & (idx < first_row + n_local)
    src = torch.from_numpy(idx[mine] - first_row).to(env.dev)
    dst = torch.from_numpy(np.nonzero(mine)[0]).to(env.dev)
    arrays = {}
    for r in range(DUMP_BATCHES):
        for t, o in zip(targets, out_ring[r]):
            a = torch.zeros((DUMP_ROWS, o.shape[1]), dtype=torch.float32, device=env.dev)
            a[dst] = o.index_select(0, src)
            if env.world > 1:
                env.dist.all_reduce(a)          # every sampled row lives on exactly one rank: the sum is that rank's row
            arrays[f"{t}_batch{r}"] = a
    if env.rank == 0:
        os.makedirs(out_dir, exist_ok=True)
        np.save(os.path.join(out_dir, "rows.npy"), idx.astype(np.float64))
        for name, a in arrays.items():
            np.save(os.path.join(out_dir, name + ".npy"), a.cpu().numpy())
    env.barrier()


# ---------------------------------------------------------------------------------------------- headline: Alarm VE
def bench_alarm_ve(env, args):
    torch = env.torch
    from continuousbayesiannetwork_b200 import sharding, synth
    from continuousbayesiannetwork_b200.engine import bind_inference, sample_network, tables_from_spec

    spec = synth.alarm()
    dev, world, rank = env.dev, env.world, env.rank
    # CPTs: 1e7 forward samples sharded over the ranks, counted on the GPU, one int64 all-reduce
    n_fit = 10_000_000
    s, e = sharding.shard_range(n_fit, rank, world)
    tables = tables_from_spec(spec, dev)
    fit_codes = sample_network(spec, seed=1236, first=s, n=e - s, device=dev, tables=tables)
    sharding.fit_sharded(tables, fit_codes, e - s)
    del fit_codes
    infer = bind_inference(tables)
    evn, tgs = synth.ALARM_EVIDENCE, synth.ALARM_TARGETS
    ids = [spec.names.index(x) for x in evn]
    s, e = sharding.shard_range(ALARM_ROWS, rank, world)
    rows = e - s
    t0 = time.perf_counter()
    plans = [infer.plan(t, evn) for t in tgs]
    fused = infer.fused_plan(tgs, evn)
    torch.cuda.synchronize()
    compile_ms = (time.perf_counter() - t0) * 1e3
    fused.set_static_evidence(True)           # resident batches replayed from a graph: nothing writes the evidence
    bpr = fused.algorithmic_bytes_per_row()
    # at least three distinct resident batches (evidence + posteriors): together they exceed 2 x L2 at every N, and the step
    # graph can keep three independent launches in flight
    ring = max(3, -(-2 * L2_BYTES // (rows * bpr)))
    ev_ring, out_ring = [], []
    for r in range(ring):
        # evidence rows drawn from the joint: forward samples; batch r of the ring is a distinct 16M-row batch
        full = sample_network(spec, seed=777 + r, first=s, n=rows, device=dev, tables=tables)
        ev_ring.append(full[ids].contiguous())
        del full
        out_ring.append([torch.empty((rows, p.card_t), dtype=torch.float32, device=dev) for p in plans])

    def one_pass(i):
        fused.run_codes(ev_ring[i % ring], rows, outs=out_ring[i % ring])

    P, est = env.passes_per_step(one_pass, args.steps, ring)
    # passes of a step are independent launches on distinct ring batches: like the Asia and 200-node legs, the step graph spreads
    # them over 3 streams, so the fill and tail of one launch hide behind its neighbour (N=8, 20 us launches on 2M-row shards:
    # +10 %; N=1, 147 us launches: +3 %); the same step on ONE stream is timed as well and reported as roofline.one_stream
    n_streams = max(1, min(3, ring))
    step_graph = env.graph_of([(lambda j=j: one_pass(j)) for j in range(P)], streams=n_streams)
    sampler = ClockSampler(env.local) if rank == 0 else None
    for _ in range(args.warmup):
        step_graph.replay()
    env.barrier()
    if sampler:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        step_graph.replay()
    e1.record()
    torch.cuda.synchronize()
    q_s = env.max_over_ranks(e0.elapsed_time(e1) / 1e3)
    clocks = sampler.stop() if sampler else None
    env.barrier()
    if args.dump_outputs:            # before any later leg writes into the ring's posteriors
        dump_headline_outputs(env, args.dump_outputs, out_ring, tgs, s)
    launches = args.steps * P
    value = ALARM_ROWS * len(tgs) * launches / q_s
    roof = roofline(env, rows * bpr, q_s / launches, "gather_tiles_kernel<2,4>" if rows >= (1 << 21) else "gather_inter_kernel<2,4>",
                    extra={"kernel_note": "4 binary targets fused, interleaved table [configuration][target][t] (27 MB, L2-resident); "
                                          "batches >= 2^21 rows take the TMA tile-staged kernel",
                           "algorithmic_bytes_per_row": bpr, "timed_region_s": q_s, "launches_in_region": launches,
                           "streams_in_step_graph": n_streams})
    if n_streams > 1:        # the same step on ONE stream, reported beside the headline figure
        g1 = env.graph_of([(lambda j=j: one_pass(j)) for j in range(P)])
        one_s = env.timed(lambda i: g1.replay(), max(3, args.steps // 4), 2) / (max(3, args.steps // 4) * P)
        roof["one_stream"] = {"launch_us": one_s * 1e6, "frac": rows * bpr / one_s / 1e9 / env.peak}
        del g1

    # ---- e2e through the C ABI with HOST buffers (pinned): H2D, kernel, D2H inside the timed region
    host_ev = ev_ring[0].cpu().pin_memory()
    host_out = [torch.empty((rows, p.card_t), dtype=torch.float32).pin_memory() for p in plans]
    e2e_steps = max(3, min(args.steps, 8))
    e2e_s = env.host_timed(lambda i: fused.run_codes_host(host_ev, rows, host_out), e2e_steps, 2)
    e2e_value = ALARM_ROWS * len(tgs) * e2e_steps / e2e_s
    fused.run_codes(ev_ring[0], rows, outs=out_ring[0])
    assert torch.equal(host_out[0], out_ring[0][0].cpu()), "host-buffer call and device path disagree"
    h2d, d2h = len(evn) * ALARM_ROWS, sum(p.card_t for p in plans) * 4 * ALARM_ROWS
    # the same call with the compact host format (CBN_HOST_OUT_DROP_LAST: card - 1 values per row travel; an API option, not
    # the reference's output format, so it is reported beside the headline e2e, not as it)
    host_c = [torch.empty((rows, p.card_t - 1), dtype=torch.float32).pin_memory() for p in plans]
    c_s = env.host_timed(lambda i: fused.run_codes_host(host_ev, rows, host_c, compact=True), e2e_steps, 2)
    assert torch.equal(host_c[0][:, 0], host_out[0][:, 0])

    # ---- e2e through the reference-facing Python API: infer(target, {name: float32 [nq,1]}) per target
    api_rows = min(rows, args.api_rows)
    f_ev = {nm: host_ev[k, :api_rows].to(torch.float32).reshape(-1, 1).pin_memory() for k, nm in enumerate(evn)}
    api_out = [torch.empty((api_rows, p.card_t), dtype=torch.float32).pin_memory() for p in plans]

    def api_step(_i):
        for tname, o in zip(tgs, api_out):
            o.copy_(infer.infer(tname, f_ev), non_blocking=True)
        torch.cuda.synchronize()

    api_s = env.host_timed(api_step, 3, 1)
    api_value = api_rows * world * len(tgs) * 3 / api_s
    assert torch.equal(api_out[0], host_out[0][:api_rows])

    def many_step(_i):
        res = infer.infer_many(tgs, f_ev)
        for tname, o in zip(tgs, api_out):
            o.copy_(res[tname], non_blocking=True)
        torch.cuda.synchronize()

    many_s = env.host_timed(many_step, 3, 1)
    many_value = api_rows * world * len(tgs) * 3 / many_s
    e2e = {"value": e2e_value, "unit": "queries/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
           "steps": e2e_steps, "pcie_GBs_per_gpu": (h2d + d2h) / world * e2e_steps / e2e_s / 1e9,
           "call": "cbn_ve_run_codes_host_multi (pinned host uint8 codes in, 4 pinned host fp32 posteriors out), one call per step over the rank's shard of the 16M-row batch",
           "timing": "host clock around the synchronous calls, barrier + synchronize on both sides, max over ranks",
           "compact": {"value": ALARM_ROWS * len(tgs) * e2e_steps / c_s, "unit": "queries/s", "h2d_bytes_per_step": h2d,
                       "d2h_bytes_per_step": sum(p.card_t - 1 for p in plans) * 4 * ALARM_ROWS,
                       "call": "cbn_ve_run_codes_host_multi_ex(..., CBN_HOST_OUT_DROP_LAST): card - 1 probabilities per row travel to the host"},
           "python_api": {"value": api_value, "unit": "queries/s", "rows_per_gpu": api_rows,
                          "pcie_GBs_per_gpu": (4 * len(evn) * api_rows * len(tgs) + d2h // ALARM_ROWS * api_rows) * 3 / api_s / 1e9,
                          "h2d_bytes_per_step": 4 * len(evn) * api_rows * len(tgs) * world, "d2h_bytes_per_step": d2h // ALARM_ROWS * api_rows * world,
                          "call": "ExactInference.infer(target, {name: pinned float32 [nq,1]}) per target -> pinned host copy (the reference's call; "
                                  "float evidence is uploaded once per target)"},
           "python_api_many": {"value": many_value, "unit": "queries/s", "rows_per_gpu": api_rows,
                               "call": "ExactInference.infer_many(targets, evidence): evidence uploaded and encoded once, one fused launch"}}
    cfg = {}
    cfg.update({"rows_per_gpu_per_pass": rows, "passes_per_step": P,
                "step": f"{P} consecutive passes over the rank's shard of a 16M-row batch (one pass = {est * 1e6:.0f} us: K steps cover >= {MIN_REGION_S * 1e3:.0f} ms)",
                "l2": (f"one batch (evidence + posteriors) is {rows * bpr / 1e6:.0f} MB per GPU > 126 MB L2" if ring == 1 else
                       f"passes rotate through a ring of {ring} distinct batches, {ring * rows * bpr / 1e6:.0f} MB per GPU > 2 x 126 MB L2"),
                "launch": (f"1 fused kernel per pass; one step = one CUDA-graph replay, passes spread over {n_streams} stream(s) inside the graph "
                           "(programmatic dependent launch between the passes of a stream)"),
                "fit": f"CPTs counted on the GPU from {n_fit} forward samples (sharded over the ranks, one int64 all-reduce)",
                "plan_compile_ms": compile_ms, "table_cells": [p.stats.final_tables[0][1] for p in plans],
                "cpu_affinity": {"visible_cpus": len(env.cpus_before or []), "bound_cpus": len(env.cpus_bound or [])}})
    res = {"value": value, "q_s": q_s, "launches": launches, "roofline": roof, "e2e": e2e, "clocks": clocks, "run_detail": cfg,
           "passes_per_step": P}
    # fused MAP prediction (benchmarking_df path): one float per row instead of a posterior row
    mplan = plans[0]
    mouts = [torch.empty(rows, dtype=torch.float32, device=dev) for _ in range(ring)]
    mplan.set_static_evidence(True)
    # 12 launches per replay over the ring's batches, three streams inside the graph like the headline; 5 replays = 60
    # launches are timed and `sec` is scaled to the 20 launches the formulas below are written for
    g = env.graph_of([(lambda j=j: mplan.run_codes_map(ev_ring[j % ring], rows, out=mouts[j % ring])) for j in range(12)], streams=n_streams)
    sec = env.timed(lambda i: g.replay(), 5, 2) / 3
    mbytes = rows * (len(mplan.stats.relevant_evidence) + 4)
    res["alarm_map"] = {"metric": "MAP predictions/sec (fused posterior + argmax + domain lookup)", "value": ALARM_ROWS * 20 / sec,
                        "unit": "rows/s", "target": tgs[0], "roofline": roofline(env, mbytes, sec / 20, "gather_tiles_kernel<2,0> (MAP epilogue)")}
    del ev_ring, out_ring, host_ev, host_out
    torch.cuda.empty_cache()
    return res


# ---------------------------------------------------------------------------------------------- config 2: Asia
def bench_asia(env, args):
    torch = env.torch
    from continuousbayesiannetwork_b200 import sharding, synth
    from continuousbayesiannetwork_b200.engine import bind_inference, sample_network, tables_from_spec

    spec = synth.asia()
    dev, world, rank = env.dev, env.world, env.rank
    out = {}
    # fit throughput: 2^28 resident samples per GPU (2 GB of codes >> L2), count + int64 all-reduce + CPTs per step
    n_big = args.fit_samples
    big = tables_from_spec(spec, dev)
    codes = sample_network(spec, seed=1235, first=rank * n_big, n=n_big, device=dev, tables=big)

    def fit_step(_i):
        big.reset_counts()
        sharding.fit_sharded(big, codes, n_big)

    k = max(3, min(args.steps, 10))
    sec = env.timed(fit_step, k, 2)
    check = verify_sharded_fit(env, spec, big, 1235, n_big) if world > 1 else None
    rate = n_big * world * k / sec
    out["fit"] = {"metric": "CPT-fit samples/sec", "value": rate, "unit": "samples/s", "samples_per_gpu_per_step": n_big, "n_vars": spec.n,
                  "table_updates_per_sample": big.count_updates_per_sample(), "includes": "count kernel + int64 all-reduce + CPT normalisation",
                  "roofline": roofline(env, n_big * spec.n, sec / k, "count_tiles_kernel (asia)"), "sharded_fit_check": check}
    del codes, big
    torch.cuda.empty_cache()
    # fit end to end from pinned HOST codes: chunked H2D overlapped with counting, then CPTs
    n_h = 1 << 26
    th = tables_from_spec(spec, dev)
    hcodes = sample_network(spec, seed=98, first=rank * n_h, n=n_h, device=dev, tables=th).cpu().pin_memory()

    def hstep(_i):
        th.reset_counts()
        th.count_host(hcodes, n_h)
        th.finalize()

    el = env.host_timed(hstep, 3, 1)
    out["fit"]["e2e"] = {"value": n_h * world * 3 / el, "unit": "samples/s", "h2d_bytes_per_step": n_h * spec.n * world, "d2h_bytes_per_step": 0,
                         "pcie_GBs_per_gpu": n_h * spec.n * 3 / el / 1e9, "call": "cbn_count_run_host + cbn_cpt_from_plan_dev (pinned host codes in, tables stay on the device)"}
    del hcodes, th
    # float32 ingestion: columns resident on the device -> domains -> codes -> counts -> CPTs (BayesianNetwork(dag, data) path)
    from continuousbayesiannetwork_b200.tables import DiscreteTables

    n_in = 1 << 26
    t0_ = tables_from_spec(spec, dev)
    c_ = sample_network(spec, seed=99, first=rank * n_in, n=n_in, device=dev, tables=t0_)
    cols = {nm: (c_[i, :n_in].to(torch.float32) * 0.5 - 1.0) for i, nm in enumerate(spec.names)}
    del c_, t0_
    ing = DiscreteTables(spec.names, spec.parents_by_name(), device=dev)
    sec = env.timed(lambda i: ing.fit_columns(cols), 5, 2)
    out["ingest_fit_f32"] = {"metric": "CPT-fit samples/sec from float32 columns (domain discovery + encoding + counting + CPTs)",
                             "value": n_in * world * 5 / sec, "unit": "samples/s", "rows_per_gpu": n_in, "n_vars": spec.n,
                             "roofline": roofline(env, n_in * spec.n * 10, sec / 5, "domain_scan + encode_f32 + count_tiles",
                                                  extra={"bytes_per_value": "4 (domain scan) + 4 + 1 (encode) + 1 (count)"})}
    del cols, ing
    torch.cuda.empty_cache()
    # queries: 1,048,576 rows per GPU, 3 fused targets; ring of distinct batches larger than 2 x L2
    n_fit = 10_000_000
    s, e = sharding.shard_range(n_fit, rank, world)
    tables = tables_from_spec(spec, dev)
    fc = sample_network(spec, seed=1235, first=s, n=e - s, device=dev, tables=tables)
    sharding.fit_sharded(tables, fc, e - s)
    del fc
    infer = bind_inference(tables)
    rows = 1 << 20
    fused = infer.fused_plan(ASIA_TARGETS, ASIA_EVIDENCE)
    fused.set_static_evidence(True)
    bpr = fused.algorithmic_bytes_per_row()
    ring = max(2, -(-2 * L2_BYTES // (rows * bpr)))
    ids = [spec.names.index(x) for x in ASIA_EVIDENCE]
    ev_ring, out_ring = [], []
    for r in range(ring):
        full = sample_network(spec, seed=4321, first=(rank * ring + r) * rows, n=rows, device=dev, tables=tables)
        ev_ring.append(full[ids].contiguous())
        out_ring.append([torch.empty((rows, 2), dtype=torch.float32, device=dev) for _ in ASIA_TARGETS])
    del full

    def one_pass(i):
        fused.run_codes(ev_ring[i % ring], rows, outs=out_ring[i % ring])

    k = max(3, min(args.steps, 20))
    P, est = env.passes_per_step(one_pass, k, ring)
    res = {}
    for streams in (1, 3):
        g = env.graph_of([(lambda j=j: one_pass(j)) for j in range(P)], streams=streams)
        sec = env.timed(lambda i: g.replay(), k, 3)
        res[streams] = sec / (k * P)
        del g
    best = min(res.values())
    out["ve"] = {"metric": METRIC, "value": rows * len(ASIA_TARGETS) * world / best, "unit": "queries/s", "rows_per_gpu_per_pass": rows,
                 "targets": 3, "passes_per_step": P, "timed_region_s": best * k * P,
                 "l2": f"ring of {ring} distinct batches, {ring * rows * bpr / 1e6:.0f} MB > 2 x 126 MB L2",
                 "roofline": roofline(env, rows * bpr, best, "gather_inter_kernel<2,3>",
                                      extra={"one_stream": {"launch_us": res[1] * 1e6, "frac": rows * bpr / res[1] / 1e9 / env.peak},
                                             "three_streams": {"launch_us": res[3] * 1e6, "frac": rows * bpr / res[3] / 1e9 / env.peak},
                                             "note": "launch-latency scale (29 MB per launch): passes of a step are one graph; with 3 streams inside the "
                                                     "graph the launch overhead of pass i+1 hides behind pass i"})}
    host_ev = [x.cpu().pin_memory() for x in ev_ring[:2]]
    host_out = [[torch.empty((rows, 2), dtype=torch.float32).pin_memory() for _ in ASIA_TARGETS] for _ in range(2)]
    el = env.host_timed(lambda i: fused.run_codes_host(host_ev[i % 2], rows, host_out[i % 2]), 20, 3)
    fused.run_codes(ev_ring[0], rows, outs=out_ring[0])
    assert torch.equal(host_out[0][0], out_ring[0][0].cpu())
    out["ve"]["e2e"] = {"value": rows * 3 * world * 20 / el, "unit": "queries/s", "h2d_bytes_per_step": 4 * rows * world,
                        "d2h_bytes_per_step": 3 * rows * 8 * world, "call": "cbn_ve_run_codes_host_multi, pinned host buffers"}
    f_ev = {nm: host_ev[0][k_, :rows].to(torch.float32).reshape(-1, 1).pin_memory() for k_, nm in enumerate(ASIA_EVIDENCE)}
    api_out = [torch.empty((rows, 2), dtype=torch.float32).pin_memory() for _ in ASIA_TARGETS]

    def api_step(_i):
        for tname, o in zip(ASIA_TARGETS, api_out):
            o.copy_(infer.infer(tname, f_ev), non_blocking=True)
        torch.cuda.synchronize()

    el = env.host_timed(api_step, 5, 1)
    out["ve"]["e2e"]["python_api"] = {"value": rows * 3 * world * 5 / el, "unit": "queries/s",
                                      "call": "ExactInference.infer(target, {name: pinned float32 [nq,1]}) per target"}
    del ev_ring, out_ring
    torch.cuda.empty_cache()
    return out


# ---------------------------------------------------------------------------------------------- config 3 fit half
def bench_alarm_fit(env, args):
    from continuousbayesiannetwork_b200 import sharding, synth
    from continuousbayesiannetwork_b200.engine import sample_network, tables_from_spec

    spec = synth.alarm()
    n = 2 * args.fit_chunk
    t = tables_from_spec(spec, env.dev)
    codes = sample_network(spec, seed=1236, first=env.rank * n, n=n, device=env.dev, tables=t)

    def step(_i):
        t.reset_counts()
        sharding.fit_sharded(t, codes, n)

    k = max(3, min(args.steps, 10))
    sec = env.timed(step, k, 2)
    check = verify_sharded_fit(env, spec, t, 1236, n) if env.world > 1 else None
    rate = n * env.world * k / sec
    return {"metric": "CPT-fit samples/sec", "value": rate, "unit": "samples/s", "n_vars": spec.n, "samples_per_gpu_per_step": n,
            "table_updates_per_sample": t.count_updates_per_sample(), "includes": "count kernel + int64 all-reduce + CPT normalisation",
            "roofline": roofline(env, n * spec.n, sec / k, "count_tiles_kernel (alarm)"), "sharded_fit_check": check}


# ---------------------------------------------------------------------------------------------- config 4: 200-node DAG
def bench_ktree200(env, args):
    torch = env.torch
    import numpy as np

    from continuousbayesiannetwork_b200 import sharding, synth
    from continuousbayesiannetwork_b200.engine import bind_inference, sample_network, tables_from_spec

    spec = synth.random_ktree_dag()
    dev, world, rank = env.dev, env.world, env.rank
    out = {}
    # ---- fit at the configuration's size: 1e9 samples in total, sample-sharded; each rank walks its shard in resident
    # blocks (generated on the device, counter-based: block b of rank r = samples [r*per + b*blk, ...)); counting is timed
    # with CUDA events block by block (generation is not part of the path), the tables accumulate, ONE all-reduce at the end
    total = args.ktree_samples
    per = (total + world - 1) // world
    per = (per + 15) // 16 * 16
    blk = min(per, args.ktree_block)
    t = tables_from_spec(spec, dev)
    buf = t.new_code_matrix(blk)
    first = rank * per
    mine = max(0, min(per, total - first))
    ms, done = 0.0, 0
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    env.barrier()
    wall0 = time.perf_counter()
    while done < mine:
        m = min(blk, mine - done)
        sample_network(spec, seed=1237, first=first + done, n=m, device=dev, tables=t, out=buf)
        e0.record()
        sharding.count_local(t, buf, m)
        e1.record()
        torch.cuda.synchronize()
        ms += e0.elapsed_time(e1)
        done += m
    e0.record()
    sharding.reduce_and_finalize(t)
    e1.record()
    torch.cuda.synchronize()
    reduce_ms = e0.elapsed_time(e1)
    wall = time.perf_counter() - wall0
    sec = env.max_over_ranks((ms + reduce_ms) / 1e3)
    env.barrier()
    assert t.n_total == total, (t.n_total, total)
    # totals and shared marginals of the global tables (size-independent properties; the oracle parity of a prefix is in tests/)
    marg, ok = {}, True
    for i, name in enumerate(spec.names):
        tab = t.table_view(t.counts, name)
        ok &= int(tab.sum()) == total
        for ax, v in enumerate(spec.parents[i] + [i]):
            m_ = tab.sum(dim=[d for d in range(tab.dim()) if d != ax]) if tab.dim() > 1 else tab
            if v in marg:
                ok &= bool(torch.equal(marg[v], m_))
            else:
                marg[v] = m_
    assert ok, "count tables of the 1e9-sample fit violate totals / shared marginals"
    rate = total / sec
    out["fit"] = {"metric": "CPT-fit samples/sec", "value": rate, "unit": "samples/s", "n_vars": spec.n, "samples_total": total,
                  "samples_per_gpu": mine, "resident_block_samples": blk, "all_reduce_ms": reduce_ms, "family_groups": t.count_groups(),
                  "table_updates_per_sample": t.count_updates_per_sample(), "wall_s_incl_generation": wall,
                  "checks": "every family table sums to the sample total; families sharing a variable agree on its marginal",
                  "includes": "count kernels over the rank's shard (block by block) + ONE int64 all-reduce + CPT normalisation",
                  "roofline": roofline(env, mine * spec.n, sec, "count_tiles_kernel (ktree200)",
                                       extra={"launch_note": "achieved = the rank's whole shard (all block launches) over the summed kernel time"})}
    del buf
    torch.cuda.empty_cache()
    # ---- queries: 8 patterns = random target + 10 random evidence variables, 1,048,576 rows each (per GPU).  Every pattern
    # rotates through its own ring of distinct batches (evidence + posteriors of one batch: 26 MB; ring of 6 > L2).
    infer = bind_inference(t, profile_compile=True)          # CUDA events around every contraction: contraction_gpu_ms
    rng = np.random.default_rng(1240)
    rows, n_ring = 1 << 20, 6
    fulls = [sample_network(spec, seed=1241 + r, first=rank * rows, n=rows, device=dev, tables=t) for r in range(n_ring)]
    t0 = time.perf_counter()
    pats = []
    for _ in range(8):
        vs = [int(v) for v in rng.choice(spec.n, size=11, replace=False)]
        plan = infer.plan(spec.names[vs[0]], [spec.names[v] for v in vs[1:]])
        plan.set_static_evidence(True)
        pats.append((plan, None, None, vs))
    torch.cuda.synchronize()
    compile_ms = (time.perf_counter() - t0) * 1e3
    rings = [[(f[vs[1:]].contiguous(), torch.empty((rows, plan.card_t), dtype=torch.float32, device=dev)) for f in fulls]
             for plan, _, _, vs in pats]
    del fulls

    def launch(pi, j):
        ev, o = rings[pi][j % n_ring]
        pats[pi][0].run_codes(ev, rows, out=o)

    def one_pass(j):
        for pi in range(len(pats)):
            launch(pi, j)

    k = max(3, min(args.steps, 10))
    P, est = env.passes_per_step(one_pass, k, n_ring)
    # Two orders of the same P x 8 launches of a step.  pass-major: the 8 patterns of a pass back to back -- their eight
    # 16 MB tables (128 MB) cycle through the 126 MB L2.  pattern-major: all P batches of one pattern back to back (what a
    # server that batches queries by plan does) -- the pattern's table stays L2-resident while distinct batches stream by.
    # Independent launches are spread over a few streams inside the step graph, as a serving loop would.
    orders = {"pass_major": [(pi, j) for j in range(P) for pi in range(len(pats))],
              "pattern_major": [(pi, j) for pi in range(len(pats)) for j in range(P)]}
    per_pass = {}
    for oname, order in orders.items():
        for streams in (1, 4):
            g = env.graph_of([(lambda pi=pi, j=j: launch(pi, j)) for pi, j in order], streams=streams)
            per_pass[f"{oname}_{streams}s"] = env.timed(lambda i: g.replay(), k, 2) / (k * P)
            del g
    best_key = min(per_pass, key=per_pass.get)
    best = per_pass[best_key]
    alg = sum(rows * p.algorithmic_bytes_per_row() for p, _, _, _ in pats)
    q = rows * len(pats) * world / best
    out["ve"] = {"metric": METRIC, "value": q, "unit": "queries/s", "rows_per_gpu_per_pattern": rows, "patterns": len(pats),
                 "passes_per_step": P, "schedule": best_key, "plan_compile_ms_total": compile_ms,
                 "l2": f"every pattern rotates through {n_ring} distinct batches of 26 MB (evidence + posteriors), {n_ring * 26 * len(pats)} MB in all",
                 "queries_per_s_incl_compile_one_pass": rows * len(pats) * world / (compile_ms / 1e3 + best),
                 "table_cells": [[c for _, c in p.stats.final_tables] for p, _, _, _ in pats],
                 "contraction_madds": [p.stats.contraction_madds for p, _, _, _ in pats],
                 "contraction_gpu_ms": [round(p.stats.contraction_gpu_ms, 3) for p, _, _, _ in pats],
                 "contraction_note": "every elimination step contracts ONE variable (sum over its <= 4 values here): arithmetic intensity is "
                                     "sum_card x n_inputs multiply-adds per output cell written, so the steps are bound by index arithmetic and by "
                                     "writing their output tables, not by floating-point throughput -- no step is a dense GEMM-shaped contraction "
                                     "that tensor cores could speed up",
                 "roofline": roofline(env, alg, best, "gather_tiles_kernel<4,0> x 8 patterns",
                                      extra={"launch_note": "one 'launch' = the 8 pattern launches of a pass (1M rows each, one 16 MB table per pattern)",
                                             "schedules": {kk: {"pass_us": v * 1e6, "frac": alg / v / 1e9 / env.peak} for kk, v in per_pass.items()}})}
    out["_keep"] = (spec, t, infer, pats)
    return out


# ---------------------------------------------------------------------------------------------- config 5: layered DAG
def bench_layered(env, args):
    torch = env.torch
    import numpy as np

    from continuousbayesiannetwork_b200 import synth
    from continuousbayesiannetwork_b200.engine import install_cpts, sample_network
    from continuousbayesiannetwork_b200.ve import PlanTooLarge, RowPlan

    dev, world, rank = env.dev, env.world, env.rank
    spec = synth.layered_dag()
    tables, infer = install_cpts(spec, dev)
    # (a) the 64 uniformly random patterns of the survey: how many can be answered exactly at all
    rng = np.random.default_rng(1241)
    n_ok = 0
    t0 = time.perf_counter()
    for _ in range(64):
        kk = int(rng.integers(5, 51))
        vs = [int(v) for v in rng.choice(spec.n, size=kk + 1, replace=False)]
        try:
            infer.compiler.compile(spec.names[vs[0]], [spec.names[v] for v in vs[1:]], dry=True)
            n_ok += 1
        except PlanTooLarge:
            pass
    random_ms = (time.perf_counter() - t0) * 1e3
    # (b) the tractable family: 64 patterns drawn the same way inside the first five layers; 1,048,576 rows per pattern
    # in total (64M queries), row-sharded over the ranks
    rows_total = args.layered_rows
    rows = (rows_total + world - 1) // world
    full = sample_network(spec, seed=1244, first=rank * rows, n=rows, device=dev, tables=tables)
    rng = np.random.default_rng(1242)
    pats, n_rowplans = [], 0
    t0 = time.perf_counter()
    for _ in range(64):
        kk = int(rng.integers(5, 51))
        vs = [int(v) for v in rng.choice(5 * 50, size=kk + 1, replace=False)]
        try:
            plan = infer.plan(spec.names[vs[0]], [spec.names[v] for v in vs[1:]])
        except PlanTooLarge:
            continue
        n_rowplans += isinstance(plan, RowPlan)
        pats.append((plan, full[vs[1:]].contiguous(), torch.empty((rows, plan.card_t), dtype=torch.float32, device=dev)))
    torch.cuda.synchronize()
    compile_ms = (time.perf_counter() - t0) * 1e3
    del full
    row_pats = [x for x in pats if isinstance(x[0], RowPlan)]
    gat_pats = [x for x in pats if not isinstance(x[0], RowPlan)]
    row_madds = sum(p.stats.per_row_madds for p, _, _ in row_pats)
    row_slice_bytes = sum(4 * p.stats.per_row_slice_cells + len(p.stats.relevant_evidence) + 4 * p.card_t for p, _, _ in row_pats)

    def run(ps):
        def f(_i=0):
            for plan, ev, o in ps:
                plan.run_codes(ev, rows, out=o)
        return f

    row_sec = env.timed(lambda i, g=env.graph_of([run(row_pats)]): g.replay(), 2, 1) / 2 if row_pats else 0.0
    gat_sec = env.timed(lambda i, g=env.graph_of([run(gat_pats)]): g.replay(), 3, 1) / 3 if gat_pats else 0.0
    sec = row_sec + gat_sec
    alg = sum(rows * p.algorithmic_bytes_per_row() for p, _, _ in pats)
    return {"metric": METRIC, "value": rows * world * len(pats) / sec, "unit": "queries/s",
            "rows_total_per_pattern": rows * world, "rows_per_gpu_per_pattern": rows, "queries_total_per_pass": rows * world * len(pats),
            "uniform_random_patterns": {"attempted": 64, "compiled": n_ok, "planner_ms_total": random_ms,
                                        "note": "induced width of the hidden part is 2^43+ cells for 63 of 64 patterns (DESIGN.md section 5): exact inference is out of reach for any order"},
            "first_five_layers_patterns": {"attempted": 64, "compiled": len(pats), "gather_plans": len(gat_pats), "per_row_plans": n_rowplans,
                                           "plan_compile_ms_total": compile_ms},
            "gather_plans": {"ms_per_pass": gat_sec * 1e3, "queries_per_s": rows * world * len(gat_pats) / gat_sec if gat_sec else None},
            "per_row_plans": {"plans": len(row_pats), "multiply_adds_per_row_all_plans": row_madds, "ms_per_pass": row_sec * 1e3,
                              "queries_per_s": rows * world * len(row_pats) / row_sec if row_sec else None,
                              "achieved_Gmadd_s_per_gpu": (row_madds * rows / row_sec / 1e9) if row_sec else None,
                              "fp32_fma_peak_Gmadd_s": 37000,
                              "bytes_read_per_row_all_plans": row_slice_bytes,
                              "slice_traffic_GBs_per_gpu": (row_slice_bytes * rows / row_sec / 1e9) if row_sec else None,
                              "slice_traffic_frac_of_hbm_peak": (row_slice_bytes * rows / row_sec / 1e9 / env.peak) if row_sec else None,
                              "note": "a per-row plan reads, for every evidence row, one contiguous slice of each static table (the cells left "
                                      "after fixing the row's evidence codes: 24-4866 floats per table set) from L2 / HBM: that slice traffic, not the "
                                      "|E| + 4*card_T bytes of the gather plans, is what the executor moves"},
            "roofline": roofline(env, alg, sec, "gather_* + ve_rows_* over the compiled patterns",
                                 extra={"bound_note": "compute-shaped: the per-row plans eliminate 1-9 hidden variables per row; see per_row_plans.achieved_Gmadd_s_per_gpu"})}


# ---------------------------------------------------------------------------------------------- config 1: FrozenLake
def bench_frozenlake(env, args):
    """BASELINE.json configs[0] through the reference-facing API: BayesianNetwork(dag, DataFrame) fit + infer on the 10,000
    fixture rows and on the 100x100 (obs, action) linspace grid of tests/test_frozen_lake_parameter_learning.py:30-33; the
    oracle's restatement of the reference's own arithmetic (fit_mle, infer_star) timed beside it on the host cores."""
    torch = env.torch
    import networkx as nx
    import numpy as np
    import pandas as pd

    from continuousbayesiannetwork_b200 import BayesianNetwork
    from oracle import cbn_oracle as O

    g = np.load(os.path.join(ROOT, "tests", "golden", "frozen_lake.npz"), allow_pickle=False)
    data = g["data"]
    df = pd.DataFrame(data, columns=["obs_0", "action", "reward"])
    dag = nx.DiGraph()
    dag.add_edges_from([("obs_0", "reward"), ("action", "reward")])
    dev = str(env.dev)
    PL, INF = {"estimator_name": "brute_force"}, {"inference_obj": "exact"}
    bn = BayesianNetwork(dag, df, PL, INF, device=dev)            # warm-up (library load, plan caches)
    t_fit = []
    for _ in range(5):
        t0 = time.perf_counter()
        bn = BayesianNetwork(dag, df, PL, INF, device=dev)
        torch.cuda.synchronize()
        t_fit.append(time.perf_counter() - t0)
    obs, act = np.meshgrid(np.linspace(0, 15, 100, dtype=np.float32), np.linspace(0, 3, 100, dtype=np.float32), indexing="ij")
    ev_rows = {"obs_0": torch.tensor(data[:, 0:1]), "action": torch.tensor(data[:, 1:2])}
    ev_grid = {"obs_0": torch.tensor(obs.reshape(-1, 1)), "action": torch.tensor(act.reshape(-1, 1))}

    def query():
        a, _ = bn.infer("reward", ev_rows, N_max=2, normalization="global_max")
        b, _ = bn.infer("reward", ev_grid, N_max=2, normalization="global_max")
        return a.cpu(), b.cpu()

    got_rows, got_grid = query()
    t_q = []
    for _ in range(10):
        t0 = time.perf_counter()
        query()
        t_q.append(time.perf_counter() - t0)
    # CPU: the reference's arithmetic restated (oracle O1)
    cores = _cpu_threads()
    cols = {n: torch.tensor(data[:, i]) for i, n in enumerate(["obs_0", "action", "reward"])}
    fams = {"obs_0": [], "action": [], "reward": ["action", "obs_0"]}
    t_cfit, mles, doms = [], {}, {}
    for _ in range(3):
        t0 = time.perf_counter()
        for n, ps in fams.items():
            pa = torch.stack([cols[p] for p in ps]) if ps else None
            mles[n] = O.fit_mle(cols[n], pa)
            doms[n] = O.node_domains(cols[n], pa)[-1]
        t_cfit.append(time.perf_counter() - t0)
    t_cq = []
    for _ in range(3):
        t0 = time.perf_counter()
        want_rows, _ = O.infer_star(mles, doms, fams["reward"], "reward", ev_rows, 2, root_ancestors=["action", "obs_0"])
        want_grid, _ = O.infer_star(mles, doms, fams["reward"], "reward", ev_grid, 2, root_ancestors=["action", "obs_0"])
        t_cq.append(time.perf_counter() - t0)
    np.testing.assert_allclose(got_rows.numpy(), want_rows.numpy(), rtol=1e-5, atol=1e-12)
    np.testing.assert_allclose(got_grid.numpy(), want_grid.numpy(), rtol=1e-5, atol=1e-12)
    nq = 20000
    med = lambda xs: sorted(xs)[len(xs) // 2]
    return {"metric": "FrozenLake fit + query through BayesianNetwork (latency scale: 10,000 samples, 20,000 query rows)",
            "fit": {"value": 10000 / med(t_fit), "unit": "samples/s", "ms": med(t_fit) * 1e3,
                    "call": "BayesianNetwork(dag, DataFrame, ...): pandas -> one H2D copy -> domains, codes, counts, CPTs (all nodes)",
                    "cpu_baseline": {"value": 10000 / med(t_cfit), "unit": "samples/s", "ms": med(t_cfit) * 1e3, "cores": cores, "kind": "port",
                                     "sample": "oracle O1 (fit_mle + node_domains = the reference's torch.unique arithmetic) on the full 10,000-row fixture, 3 nodes"}},
            "query": {"value": nq / med(t_q), "unit": "rows/s", "ms": med(t_q) * 1e3,
                      "call": "infer('reward', {obs_0, action}, N_max=2, normalization='global_max') on the 10,000 fixture rows + the 100x100 grid, results copied to the host",
                      "e2e": {"value": nq / med(t_q), "unit": "rows/s", "h2d_bytes_per_step": nq * 8, "d2h_bytes_per_step": nq * 8},
                      "cpu_baseline": {"value": nq / med(t_cq), "unit": "rows/s", "ms": med(t_cq) * 1e3, "cores": cores, "kind": "port",
                                       "sample": "oracle O1 infer_star (the reference's get_prob broadcast join + global max) on the same 20,000 rows"},
                      "parity": "posteriors within 1e-5 of the oracle on all 20,000 rows (checked in this run)"}}


# ---------------------------------------------------------------------------------------------- driver
def run_ours(args):
    env = Env()
    from continuousbayesiannetwork_b200 import synth

    head = bench_alarm_ve(env, args)
    configs = {}
    keep = None
    if not args.no_extras:
        configs["c3_alarm"] = {"ve": "the headline (top-level value / roofline / e2e)", "fit": bench_alarm_fit(env, args),
                               "map": head.pop("alarm_map")}
        configs["c2_asia"] = bench_asia(env, args)
        kt = bench_ktree200(env, args)
        keep = kt.pop("_keep")
        configs["c4_ktree200"] = kt
        configs["c5_layered1000"] = {"ve": bench_layered(env, args)}
        if env.rank == 0 and env.world == 1:
            configs["c1_frozenlake"] = bench_frozenlake(env, args)
    else:
        head.pop("alarm_map", None)
    if env.rank == 0:
        cpu = None
        if env.world == 1 and not args.no_cpu_baseline:
            if env.cpus_before:
                os.sched_setaffinity(0, env.cpus_before)      # the CPU baselines get every host core
            spec = synth.alarm()
            net = _oracle_net_from_samples(spec, 200_000, 1236)
            cpu = cpu_ve(spec, net, synth.ALARM_EVIDENCE, synth.ALARM_TARGETS, 65536, args.cpu_budget_s, label="Alarm 16M-row")
            if configs:
                b = args.cpu_budget_s / 2
                configs["c3_alarm"]["fit"]["cpu_baseline"] = cpu_fit(spec, 200_000, b, label="Alarm")
                asia = synth.asia()
                configs["c2_asia"]["ve"]["cpu_baseline"] = cpu_ve(asia, _oracle_net_from_samples(asia, 200_000, 1235), ASIA_EVIDENCE,
                                                                 ASIA_TARGETS, 65536, b, label="Asia 1M-row")
                configs["c2_asia"]["fit"]["cpu_baseline"] = cpu_fit(asia, 1_000_000, b, label="Asia")
                kspec, _, _, pats = keep
                configs["c4_ktree200"]["fit"]["cpu_baseline"] = cpu_fit(kspec, 200_000, b, label="the 200-node DAG")
                knet = _oracle_net_from_samples(kspec, 100_000, 1237)
                vs = pats[0][3]
                configs["c4_ktree200"]["ve"]["cpu_baseline"] = cpu_ve(kspec, knet, [kspec.names[v] for v in vs[1:]], [kspec.names[vs[0]]], 2048, b,
                                                                      label="200-node DAG pattern-0")
        roof, e2e = head["roofline"], head["e2e"]
        if configs:
            pc_r, pc_c, pc_e = {}, {}, {}
            for cname, c in configs.items():
                for leg, o in c.items():
                    if not isinstance(o, dict):
                        continue
                    key = f"{cname}.{leg}"
                    if "roofline" in o:
                        pc_r[key] = {"value": o.get("value"), "unit": o.get("unit"), "frac": o["roofline"]["frac"], "achieved_GBs": o["roofline"]["achieved"]}
                    if "cpu_baseline" in o:
                        pc_c[key] = {"value": o["cpu_baseline"]["value"], "unit": o["cpu_baseline"]["unit"], "cores": o["cpu_baseline"]["cores"],
                                     "gpu_value": o.get("value")}
                    if "e2e" in o:
                        pc_e[key] = {"value": o["e2e"]["value"], "unit": o["e2e"]["unit"]}
            roof["per_config"], e2e["per_config"] = pc_r, pc_e
            if cpu is not None:
                cpu["per_config"] = pc_c
        line = {"metric": METRIC, "value": head["value"], "unit": "queries/s", "n_gpus": env.world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": head["q_s"] / args.steps * 1e3, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
                "dtype": "f32", "data": "synthetic", "config": CONFIG, "e2e": e2e, "gpu_launches": head["launches"] * env.world,
                "roofline": roof, "cpu_baseline": cpu, "clocks": head["clocks"], "run_detail": head["run_detail"], "configs": configs}
        print(json.dumps(line))
    if env.world > 1:
        env.dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--fit-chunk", type=int, default=1 << 25)
    ap.add_argument("--fit-samples", type=int, default=1 << 28)
    ap.add_argument("--ktree-samples", type=int, default=1_000_000_000)
    ap.add_argument("--ktree-block", type=int, default=1 << 27)
    ap.add_argument("--layered-rows", type=int, default=1 << 20)
    ap.add_argument("--api-rows", type=int, default=1 << 22)
    ap.add_argument("--ref-rows", type=int, default=1 << 17)
    ap.add_argument("--cpu-budget-s", type=float, default=10.0)
    ap.add_argument("--no-extras", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the headline posteriors of the last step (a fixed, seeded sample of rows) "
                         "to DIR/<target>_batch<r>.npy, with the sampled row ids in DIR/rows.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
