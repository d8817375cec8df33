#!/usr/bin/env python
"""bench.py -- LP edges/s on B200 (BASELINE.json metric) for the B200-native label-propagation
engine, next to the reference's own CPU path.

A "step" = one ``LPClustering.compute_clustering`` call (5 LP rounds + post passes,
lp_clusterer.cc:89-109) on the synthetic input, the timed region of the reference's own harness
(apps/benchmarks/shm_label_propagation_benchmark.cc:121-123).

  value  : scanned directed edges per second, graph already resident in HBM (device-timed)
  e2e    : the same through the public API with HOST buffers -- graph H2D, clustering D2H inside
           the timed region
  roofline: dominant sweep kernel family, algorithmic bytes (8 B/scanned edge + 16 B/visited
           vertex, SURVEY.md §8d) / CUDA-event time of those launches, vs MEASURED_PEAKS.json
  cpu_baseline: the unmodified reference (oracle/_ref) on all host cores (OpenMP mode of the oneTBB
           stand-in) or, when that library is absent, the oracle port, on a bounded sample

``--impl reference`` times only the CPU reference arm on the same workload definition.

``--dump-outputs DIR`` writes what the last timed step computed (the arrays a caller of the timed path receives)
to DIR/<name>.npy; the inputs are generated from fixed seeds, so two builds can be compared output for output.
The LP random draws are seeded per call (like the reference's), so the last step's result depends on
--warmup + --steps: compare runs made with the same arguments.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

WORKLOADS = {
    # name: (generator, args, k)   -- BASELINE.json configs
    "rmat22": ("rmat", dict(scale=22, edge_factor=16, seed=1), 16),   # configs[1]
    "rmat24": ("rmat", dict(scale=24, edge_factor=16, seed=1), 64),   # configs[3]
    "rmat20": ("rmat", dict(scale=20, edge_factor=16, seed=1), 16),
    "rmat18": ("rmat", dict(scale=18, edge_factor=16, seed=1), 16),
    "grid512": ("grid", dict(nx=512), 64),                             # configs[2]
    "grid256": ("grid", dict(nx=256), 64),
    "rgg24": ("rgg", dict(n=1 << 24, seed=1), 64),
    "rgg20": ("rgg", dict(n=1 << 20, seed=1), 64),
    # configs[4]: road-like planar graph, ~23 M vertices / ~56 M directed edges (SURVEY.md §8d input 5)
    "road": ("road", dict(side=3500, seed=1, delete_frac=0.3, subdivide_frac=0.65), 256),
    "road_small": ("road", dict(side=1000, seed=1, delete_frac=0.3, subdivide_frac=0.65), 256),
}
# Workload the CPU reference runs for a given GPU workload. Like for like wherever the reference finishes a
# step in about a second (R-MAT 22: ~1.3 s/step on the box's host cores); only the three largest inputs
# use a smaller graph of the same family so that `--impl reference --steps K --warmup W` (plus the thread
# sweep) still ends within a few minutes -- the line's config says so ("cpu_sample").
CPU_SAMPLE = {"rmat24": "rmat22", "grid512": "grid256", "rgg24": "rgg20", "road": "road_small"}


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def generate(name, device):
    """Synthetic input after the degree-bucket rearrangement the facade applies (kaminpar.cc:369-396).
    Returns torch int64 (xadj, adjncy) on `device`."""
    import torch

    from kaminpar_b200 import graph as G

    kind, args, k = WORKLOADS[name]
    if kind == "rmat":
        n = 1 << args["scale"]
        src, dst = G.rmat_edges_torch(args["scale"], args["edge_factor"], args["seed"], device)
        xadj, adj = G._csr_from_pairs_torch(n, src, dst, device)
    elif kind == "grid":
        xadj, adj = G.grid3d_torch(args["nx"], device)
    elif kind == "rgg":
        g = G.rgg2d(args["n"], args["seed"], device=device)
        xadj = torch.from_numpy(g.xadj.astype(np.int64)).to(device)
        adj = torch.from_numpy(g.adjncy.astype(np.int64)).to(device)
    elif kind == "road":
        g = G.road_like(args["side"], args["seed"], args["delete_frac"], args["subdivide_frac"], device=device)
        xadj = torch.from_numpy(g.xadj.astype(np.int64)).to(device)
        adj = torch.from_numpy(g.adjncy.astype(np.int64)).to(device)
    else:
        raise ValueError(kind)
    xadj, adj, _ = G.rearrange_by_degree_buckets_torch(xadj, adj, remove_isolated=True)
    return xadj, adj, k


DUMP_BUDGET_BYTES = 64 << 20


def dump_outputs(out_dir, arrays):
    """Write every array as <out_dir>/<name>.npy: float32 where each value is exact in it (|x| <= 2^24), float64
    otherwise. When the total exceeds DUMP_BUDGET_BYTES, every array larger than its share of the budget is cut to
    a sample of positions drawn with a fixed seed (the same positions for the same length in every run); the
    positions go to <name>_index.npy."""
    os.makedirs(out_dir, exist_ok=True)
    out = {}
    for name, a in arrays.items():
        a = np.asarray(a)
        out[name] = a.astype(np.float32 if a.size == 0 or np.abs(a).max() <= (1 << 24) else np.float64)
    if sum(a.nbytes for a in out.values()) > DUMP_BUDGET_BYTES:
        share = DUMP_BUDGET_BYTES // len(out)
        for name in list(out):
            a = out[name]
            if a.nbytes > share:
                idx = np.sort(np.random.default_rng(0).choice(a.size, share // (a.itemsize + 8), replace=False))
                out[name] = a[idx]
                out[name + "_index"] = idx.astype(np.float64)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index):
        self.index = index
        self.samples = []
        self.proc = None

    def start(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.samples.append((time.monotonic(), line.strip()))

    def mark_begin(self):
        """Start of the timed region (the sampler itself is started earlier: nvidia-smi needs > 100 ms to emit its
        first line, a short timed region would otherwise end with no sample)."""
        self.t_begin = time.monotonic()

    def mark_end(self):
        self.t_end = time.monotonic()

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        t0 = getattr(self, "t_begin", None)
        t1 = getattr(self, "t_end", None)
        if t0 is not None and t1 is not None and time.monotonic() - t0 < 0.35:
            time.sleep(0.35 - (time.monotonic() - t0))  # let at least one more 100 ms tick arrive
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, smax, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        lines = [s for _, s in self.samples]
        where = "whole sampled interval"
        if t0 is not None and t1 is not None:
            inside = [s for t, s in self.samples if t0 <= t <= t1 + 0.05]
            if inside:
                lines, where = inside, "timed region"
            else:  # region shorter than the sampling period: the samples next to it (same kernels before / after)
                near = [s for t, s in self.samples if t0 - 0.3 <= t <= t1 + 0.3]
                lines, where = (near or lines), "within 0.3 s of the timed region (region < sampling period)"
        for s in lines:
            parts = [p.strip() for p in s.split(",")]
            if len(parts) < 6:
                continue
            try:
                sm.append(float(parts[0]))
                smax.append(float(parts[1]))
            except ValueError:
                continue
            for nm, v in zip(names, parts[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "reasons": sorted(reasons), "samples": len(sm), "sampled": where}


def _cpu_worker(name, mode, steps, warmup, host_graph=None):
    """Run oracle/cpu_baseline_worker.py on workload `name` (or its CPU_SAMPLE stand-in) in a child process
    that never loads torch (isolation: see the worker's header). `host_graph` = (xadj, adjncy, k) numpy
    arrays of `name` itself if the caller already has them. Returns
    (units_per_s, s_per_step, kind, cores, description, extra) with extra = host cores + thread sweep."""
    import subprocess
    import tempfile

    sample = CPU_SAMPLE.get(name, name)
    if sample == name and host_graph is not None:
        xadj_np, adj_np, k = host_graph
    else:
        import torch

        # generation is not timed: use the GPU for it when there is one (same generator, same seed)
        gen_dev = "cuda" if torch.cuda.is_available() else "cpu"
        xadj, adj, k = generate(sample, gen_dev)
        xadj_np, adj_np = xadj.cpu().numpy(), adj.cpu().numpy()
        del xadj, adj
    with tempfile.TemporaryDirectory() as tmp:
        path = os.path.join(tmp, "sample.npz")
        np.savez(path, xadj=np.asarray(xadj_np).astype(np.uint32), adjncy=np.asarray(adj_np).astype(np.uint32),
                 k=np.array([k]))
        del xadj_np, adj_np
        last_err = ""
        env = dict(os.environ, OMP_STACKSIZE=os.environ.get("OMP_STACKSIZE", "64M"))
        env.pop("OMP_NUM_THREADS", None)  # torchrun exports 1; the worker sizes its team from the affinity mask
        for extra in ([], ["serial"]):  # second try: the serial stand-in (1 core), should the OpenMP one fail
            r = subprocess.run([sys.executable, "-m", "oracle.cpu_baseline_worker", path, mode, str(steps), str(warmup)]
                               + extra, cwd=ROOT, capture_output=True, text=True, env=env)
            lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
            if r.returncode == 0 and lines:
                d = json.loads(lines[-1])
                more = {"host_cores": d.get("host_cores"), "thread_sweep": d.get("thread_sweep"),
                        "workload": sample, "same_workload": sample == name}
                return d["value"], d["seconds_per_step"], d["kind"], d["cores"], f"{sample}: {d['desc']}", more
            last_err = f"rc={r.returncode} {r.stderr[-300:]}"
    raise RuntimeError("CPU baseline worker failed: " + last_err)


def cpu_reference_run(name, steps, warmup, host_graph=None):
    """The reference's own CPU path (oracle/_ref: unmodified sources on the host cores through the OpenMP
    stand-in for oneTBB; serial stand-in or the oracle port if that did not travel)."""
    return _cpu_worker(name, "lp", steps, warmup, host_graph)


def cpu_contraction_run(name, steps, warmup, host_graph=None):
    """contract_clustering of the unmodified reference (oracle/_ref) or the numpy port."""
    return _cpu_worker(name, "contraction", steps, warmup, host_graph)


def contraction_mode(args, handle, g_host, n, m, k, mcw, dev, local_rank):
    """--mode contraction: a step = one contract_clustering of the (device-resident) LP clustering."""
    import torch

    from kaminpar_b200 import contraction as KC
    from kaminpar_b200 import lp

    metric, unit = "contraction_fine_edges_per_second", "edges/s"
    handle.set_timing(False)
    handle.cluster(mcw, fetch=False)
    cl_host = handle.download_labels()
    sampler = ClockSampler(local_rank)
    sampler.start()
    for _ in range(args.warmup):
        KC.contract_on_handle(handle, None).close()
    torch.cuda.synchronize()
    sampler.mark_begin()
    tot_ms, launches, last = 0.0, 0, None
    for step in range(args.steps):
        cg = KC.contract_on_handle(handle, None)
        tot_ms += cg.stats.device_ms
        launches += cg.stats.kernel_launches
        last = (cg.stats.c_n, cg.stats.c_m, cg.stats.cut_edges, cg.stats.sort_bits)
        if args.dump_outputs is None or step + 1 < args.steps:
            cg.close()
    torch.cuda.synchronize()
    sampler.mark_end()
    if args.dump_outputs is not None:  # the coarse graph of the last timed step
        c = cg.get()
        dump_outputs(args.dump_outputs, {"c_xadj": c.xadj, "c_adjncy": c.adjncy, "c_vwgt": c.vwgt,
                                         "c_adjwgt": c.adjwgt, "mapping": cg.mapping()})
        cg.close()
    clocks = sampler.stop()
    value = m * args.steps / (tot_ms * 1e-3)
    c_n, c_m, cut, bits = last
    # e2e: graph + clustering from host memory, coarse graph + mapping back to the host
    ctx = lp.create_default_context()
    ctx.engine.device = local_rank
    e2e = None
    if not args.no_e2e:
        h2 = lp.LPHandle(lp._cluster_config(ctx.coarsening.clustering.lp, ctx.engine))

        def e2e_step():
            h2.set_graph(g_host)
            cg = KC.contract_on_handle(h2, cl_host)
            cg.get()
            cg.mapping()
            cg.close()

        e2e_step()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            e2e_step()
        torch.cuda.synchronize()
        e2e_s = time.perf_counter() - t0
        e2e = {"value": m * args.steps / e2e_s, "unit": unit, "h2d_bytes_per_step": (n + 1) * 4 + m * 4 + n * 4,
               "d2h_bytes_per_step": (c_n + 1) * 4 + c_m * 8 + c_n * 4 + n * 4, "ms_per_step": e2e_s / args.steps * 1e3}
    peak, peak_src = peaks()
    alg = 8 * m + 12 * n + 12 * c_m + 8 * c_n
    achieved = alg * args.steps / (tot_ms * 1e-3) / 1e9
    line = {
        "metric": metric, "value": value, "unit": unit, "n_gpus": 1, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": tot_ms / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "int32", "data": "synthetic",
        "config": {"workload": args.workload, "n": n, "m_directed": m, "k": k, "mode": "contraction",
                   "coarse_n": c_n, "coarse_m": c_m, "inter_cluster_edges": cut, "sort_bits": bits,
                   "l2": "inputs_larger_than_l2" if m * 4 > 126e6 else "small_input"},
        "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches),
        "roofline": {"bound": "hbm", "kernel": "contract_clustering (key pass + radix sort + reduce-by-key)",
                     "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": None,
                     "peak_source": peak_src, "algorithmic_bytes_per_launch": alg,
                     "note": "8 B per fine edge + 12 B per fine vertex + 12 B per coarse edge + 8 B per coarse vertex; "
                             "the radix passes over the inter-cluster edges are not algorithmic bytes"},
    }
    if not args.no_cpu_baseline:
        eps, dt, kind, cores, desc, more = cpu_contraction_run(args.workload, args.cpu_steps, 1,
                                                               (g_host.xadj, g_host.adjncy, k))
        line["cpu_baseline"] = {"value": eps, "unit": unit, "cores": cores, "kind": kind, "sample": desc, **more}
    print(json.dumps(line), flush=True)
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default=os.environ.get("KMP_BENCH_WORKLOAD"),
                    help="default: rmat22 (BASELINE config 2) on 1 GPU, rmat24 (config 4: R-MAT scale 24, k=64, "
                         "2/4/8 x B200) on N > 1")
    ap.add_argument("--cpu-steps", type=int, default=2)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true", help="profiling runs only: skip the host-buffer arm (e2e = null)")
    ap.add_argument("--mode", default="clustering", choices=["clustering", "refinement", "contraction"],
                    help="refinement: one LabelPropagationRefiner.refine call on a hashed k-way partition (N=1 only); "
                         "contraction: contract_clustering of the LP clustering (SURVEY §8f-1, N=1 only)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the outputs of the last timed step as DIR/<name>.npy (float32 / float64, <= 64 MB "
                         "in all): clustering; partition + block_weights; c_xadj, c_adjncy, c_vwgt, c_adjwgt, mapping")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs is not None and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the GPU path (--impl b200)")
    if args.workload is None:
        args.workload = "rmat22" if args.gpus <= 1 else "rmat24"

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    metric = "lp_edges_per_second"
    unit = "edges/s"
    _, _, k = WORKLOADS[args.workload][0], WORKLOADS[args.workload][1], WORKLOADS[args.workload][2]

    if args.impl == "reference":
        if rank != 0:
            return 0
        eps, dt, kind, cores, desc, more = cpu_reference_run(args.workload, args.steps, max(args.warmup, 1))
        print(json.dumps({
            "impl": "reference", "metric": metric, "value": eps, "unit": unit, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "int32", "data": "synthetic",
            "config": {"workload": args.workload, "k": k, "mode": "clustering",
                       "cpu_sample": more["workload"], "same_workload": more["same_workload"]},
            "cpu_baseline": {"value": eps, "unit": unit, "cores": cores, "kind": kind, "sample": desc, **more},
            "e2e": {"value": eps, "unit": unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        }), flush=True)
        # two OpenMP runtimes live in this process (torch's and the stand-in's): skip interpreter teardown
        os._exit(0)

    import torch
    import torch.distributed as dist

    from kaminpar_b200 import lp
    from kaminpar_b200.graph import CSRGraph

    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device: kaminpar_b200 has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    # ---- input (synthetic, generated on the device; per-rank seed offset for N > 1) ------------
    wl = args.workload
    xadj64, adj64, k = generate(wl, dev)
    n = xadj64.numel() - 1
    m = adj64.numel()
    d_xadj = xadj64.to(torch.int32)   # bit pattern == uint32 (m < 2^31)
    d_adj = adj64.to(torch.int32)
    del xadj64, adj64
    torch.cuda.synchronize()
    h_xadj = torch.empty(n + 1, dtype=torch.int32, pin_memory=True).copy_(d_xadj)
    h_adj = torch.empty(m, dtype=torch.int32, pin_memory=True).copy_(d_adj)
    h_out = torch.empty(n, dtype=torch.int32, pin_memory=True)
    g_host = CSRGraph.__new__(CSRGraph)  # views on pinned memory, no copies
    g_host.xadj = h_xadj.numpy().view(np.uint32)
    g_host.adjncy = h_adj.numpy().view(np.uint32)
    g_host.vwgt = None
    g_host.adjwgt = None
    g_host.sorted = True
    g_host.buckets = None

    ctx = lp.create_default_context()
    ctx.partition.setup(g_host, k, 0.03)
    mcw = lp.compute_max_cluster_weight(ctx.coarsening, ctx.partition, n, n)

    # ---- device-resident arm ("value") -------------------------------------------------------
    ctx.engine.device = local_rank
    handle = lp.LPHandle(lp._cluster_config(ctx.coarsening.clustering.lp, ctx.engine))
    handle.set_graph_device(n, m, d_xadj.data_ptr(), d_adj.data_ptr())
    # timed region: per-tier events OFF (the independent kernel tiers of a sub-round then overlap on side streams);
    # the per-tier breakdown / roofline comes from extra steps with events ON after the timed region
    handle.set_timing(False)
    if args.mode == "contraction":
        return contraction_mode(args, handle, g_host, n, m, k, mcw, dev, local_rank)
    if world > 1:
        # strong scaling: ONE graph, vertex frontier sharded over the ranks; the library all-gathers the proposal
        # buffers itself (ncclAllGather on the handle's stream, kmp_lp_dist_init) between sweep and commit
        handle.dist_init(rank, world)

    refine_handle = None
    if args.mode == "refinement":
        # SURVEY §8d refinement mode: hash-of-id blocks, max_block_weight = (1+eps)*ceil(n/k)
        refine_handle = lp.LPHandle(lp._refine_config(ctx.refinement.lp, ctx.engine))
        refine_handle.set_graph_device(n, m, d_xadj.data_ptr(), d_adj.data_ptr())
        refine_handle.set_timing(False)
        rng = np.random.default_rng(0)
        part0 = rng.integers(0, k, n).astype(np.uint32)
        mbw = ctx.partition.max_block_weights()

    sharded_moved = []  # per-round move counts of the last sharded step (identical on every rank)
    block_weights = [None]  # returned by the last refinement step

    def run_resident():
        if refine_handle is not None:
            refine_handle.upload_partition(part0)
            _, block_weights[0], st = refine_handle.refine(k, mbw, None)
            return st
        return handle.cluster(mcw, fetch=False)[1]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    sampler = ClockSampler(local_rank)
    sampler.start()
    for _ in range(args.warmup):
        run_resident()
    barrier()
    sampler.mark_begin()
    tot_ms = 0.0
    edges = nodes = launches = sweeps = 0
    NT = 8  # kernel tiers (include/kaminpar_b200_lp.h kmp_lp_stats)
    g_edges = [0] * NT
    g_nodes = [0] * NT
    g_ms = [0.0] * NT
    commit_ms = apply_ms = push_ms = 0.0
    pull_rounds = push_rounds = 0
    g_launch = [0] * NT
    last = None
    for _ in range(args.steps):
        st = run_resident()
        tot_ms += st.device_ms
        edges += st.edges_scanned
        nodes += st.nodes_visited
        launches += st.kernel_launches
        sweeps += st.sweep_launches
        pull_rounds += st.pull_rounds
        push_rounds += st.push_rounds
        last = st
    barrier()
    sampler.mark_end()
    if args.dump_outputs is not None and rank == 0:  # the labels the last timed step left on the device
        if refine_handle is not None:
            dump_outputs(args.dump_outputs, {"partition": refine_handle.download_labels(),
                                             "block_weights": block_weights[0]})
        else:
            dump_outputs(args.dump_outputs, {"clustering": handle.download_labels()})
    # ---- breakdown steps (outside the timed region): per-tier CUDA events, tiers serialised ----------------
    BSTEPS = 2
    (refine_handle or handle).set_timing(True)
    brk_ms = 0.0
    for _ in range(BSTEPS):
        st = run_resident()
        brk_ms += st.device_ms
        for q in range(NT):
            g_edges[q] += st.group_edges[q]
            g_nodes[q] += st.group_nodes[q]
            g_ms[q] += st.group_sweep_ms[q]
            g_launch[q] += st.group_launches[q]
        commit_ms += st.group_sweep_ms[12]
        apply_ms += st.group_sweep_ms[13]
        push_ms += st.group_sweep_ms[14]
    (refine_handle or handle).set_timing(False)
    barrier()
    clocks = sampler.stop()
    t = torch.tensor([tot_ms, float(edges)], dtype=torch.float64, device=dev)
    if world > 1:
        tmax = t.clone()
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        # every rank's stats already hold the whole job's scan counters (ncclAllReduce in the library)
        tot_ms_max, edges_all = float(tmax[0]), float(edges)
    else:
        tot_ms_max, edges_all = tot_ms, float(edges)
    value = edges_all / (tot_ms_max * 1e-3)

    # ---- e2e arm: public API, host buffers, H2D + D2H inside the timed region -------------------
    clusterer = lp.LPClustering(ctx.coarsening, ctx.engine)
    clusterer.set_max_cluster_weight(mcw)
    out_np = h_out.numpy().view(np.uint32)

    e2e_handle = None
    if world > 1:
        e2e_handle = lp.LPHandle(lp._cluster_config(ctx.coarsening.clustering.lp, ctx.engine))
        e2e_handle.dist_init(rank, world)

    refiner = p_graph_host = None
    if args.mode == "refinement":
        refiner = lp.LabelPropagationRefiner(ctx)
        p_graph_host = lp.PartitionedGraph(g_host, k, part0)

    def e2e_step():
        if refiner is not None:  # Refiner API: graph + partition H2D, refined partition + block weights D2H
            p_graph_host.partition[:] = part0
            refiner._graph = None
            refiner.initialize(p_graph_host)
            refiner.refine(p_graph_host, ctx.partition)
            return refiner.last_stats.edges_scanned
        if world == 1:
            clusterer._graph = None  # new graph each step: forces the H2D copy, as one coarsening level does
            clusterer.compute_clustering(g_host, clustering=out_np)
            return clusterer.last_stats.edges_scanned
        e2e_handle.set_graph(g_host)  # every rank stages its replica of the graph from pinned host memory
        _, st_e = e2e_handle.cluster(mcw, out=out_np)
        return st_e.edges_scanned

    e2e_edges = 0
    t0 = time.perf_counter()
    if not args.no_e2e:
        for _ in range(max(1, min(args.warmup, 2))):
            e2e_step()
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            e2e_edges += e2e_step()
        torch.cuda.synchronize()
    e2e_s = max(time.perf_counter() - t0, 1e-9)
    t = torch.tensor([e2e_s, float(e2e_edges)], dtype=torch.float64, device=dev)
    if world > 1:
        tmax = t.clone()
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        e2e_s = float(tmax[0])
    e2e_value = e2e_edges / e2e_s
    h2d = (n + 1) * 4 + m * 4
    d2h = n * 4
    if refiner is not None:
        h2d += n * 4 + k * 4
        d2h += k * 4

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return 0

    # ---- roofline of the dominant sweep kernel family -------------------------------------------
    peak, peak_src = peaks()
    names = ["sweep_thread<8>(deg<8)", "sweep_thread<16>(deg<=16)", "sweep_thread<32>(deg<32)",
             "sweep_team<32>(deg<256)", "sweep_team<128>(deg<1024)", "sweep_team<512>(deg<4096)", "sweep_team<1024>(deg<16384)",
             "sweep_hub_scatter+select+final(deg>=16384)"]
    dom = int(np.argmax(g_ms))
    alg_bytes = 8 * g_edges[dom] + 16 * g_nodes[dom]
    achieved = alg_bytes / (g_ms[dom] * 1e-3) / 1e9 if g_ms[dom] > 0 else 0.0
    b_edges, b_nodes = sum(g_edges), sum(g_nodes)
    all_bytes = 8 * b_edges + 16 * b_nodes
    sweep_ms_total = sum(g_ms)
    traffic = None
    try:  # DRAM bytes per launch of this kernel from the committed ncu capture (profiles/), if any
        with open(os.path.join(ROOT, "profiles", "r2_traffic.json")) as f:
            traffic = json.load(f).get(wl, {}).get(names[dom], {}).get("traffic_bytes_per_launch")
    except Exception:
        traffic = None
    roofline = {
        "bound": "hbm", "kernel": names[dom], "achieved": achieved, "peak": peak, "unit": "GB/s",
        "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src,
        "launches": g_launch[dom], "avg_launch_ms": g_ms[dom] / max(g_launch[dom], 1),
        "algorithmic_bytes_per_launch": alg_bytes / max(g_launch[dom], 1),
        "share_of_step": g_ms[dom] / brk_ms if brk_ms > 0 else None,
        "measured_in": f"{BSTEPS} extra steps after the timed region with per-tier CUDA events on (tiers of a "
                       f"sub-round serialised; {brk_ms / BSTEPS:.3f} ms/step there vs ms_per_step with the tiers overlapped)",
        "all_sweeps": {"achieved": all_bytes / (sweep_ms_total * 1e-3) / 1e9 if sweep_ms_total > 0 else 0.0,
                       "share_of_step": sweep_ms_total / brk_ms if brk_ms > 0 else None,
                       "per_group_ms": [x / BSTEPS for x in g_ms],
                       "per_group_edges": [x // BSTEPS for x in g_edges]},
        "commit_ms": commit_ms / BSTEPS, "apply_ms": apply_ms / BSTEPS, "push_activate_ms": push_ms / BSTEPS,
        "pull_rounds_per_step": pull_rounds / args.steps, "push_rounds_per_step": push_rounds / args.steps,
        "gather_bound": {
            # scripts/microbench_lsu.cu on this pool's B200: random 4-byte gathers from an L2-resident table
            # (one per scanned edge is the floor of any LP sweep on a graph without locality) run at 272 G/s
            "l2_gather_per_s": 272e9,
            "all_sweeps_frac_of_gather_bound": (b_edges / (sweep_ms_total * 1e-3) / 272e9) if sweep_ms_total > 0 else None,
        },
    }

    cpu = None
    if not args.no_cpu_baseline and world == 1:  # reported on rank 0 at N=1 only
        eps, dt, kind, cores, desc, more = cpu_reference_run(wl, args.cpu_steps, 1, (g_host.xadj, g_host.adjncy, k))
        cpu = {"value": eps, "unit": unit, "cores": cores, "kind": kind, "sample": desc, **more}

    line = {
        "metric": metric, "value": value, "unit": unit, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": tot_ms_max / args.steps, "higher_is_better": True,
        # ONE graph of fixed size for every N (the vertex frontier is sharded): total work is fixed
        "scaling": "strong", "vs_baseline": None,
        "dtype": "int32", "data": "synthetic",
        "config": {"workload": wl, "n": n, "m_directed": m, "k": k, "mode": args.mode,
                   "max_cluster_weight": mcw,
                   "iterations": last.iterations, "moved": last.moved_list(),
                   "num_clusters": last.num_clusters, "l2": "inputs_larger_than_l2" if m * 4 > 126e6 else "small_input",
                   "parallelism": "single" if world == 1 else f"frontier-sharded x{world} (replicated labels; ncclAllGather of the proposal buffers per sub-round inside the library)",
                   "subrounds": ctx.engine.sync_subrounds},
        "clocks": clocks,
        "e2e": None if args.no_e2e else {"value": e2e_value, "unit": unit, "h2d_bytes_per_step": h2d,
                                         "d2h_bytes_per_step": d2h, "ms_per_step": e2e_s / args.steps * 1e3},
        "gpu_launches": int(launches),
        "roofline": roofline,
    }
    if cpu is not None:
        line["cpu_baseline"] = cpu
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
