#!/usr/bin/env python
"""bench.py — headline benchmark of the Lux hot path on B200.

Metric (BASELINE.json): MTEPS = edges processed / second / 1e6 of pull-model PageRank on the synthetic RMAT-27
CSC graph (134,217,728 V / 2,147,483,648 E, a,b,c,d = .57/.19/.19/.05, seed 27), 1/2/4/8 B200.
A "step" = ITERS_PER_STEP (10, the reference's usual -ni) PageRank iterations over the whole graph.

  python bench.py --gpus N --steps K --warmup W            # our engine (libluxb through the C ABI)
  python bench.py --impl reference ...                      # the CPU restatement of the reference on host cores

Ours arm JSON keys: value (device-resident, CUDA events, max over ranks), e2e (host buffers through the C ABI:
H2D of the initial vertex values from pinned memory + iterations + D2H of the result, per step), roofline of the
dominant kernel (pull_tile_kernel), cpu_baseline (oracle on the box's host cores, bounded sample), clocks.
N > 1: launched by torch.distributed.run, one rank per GPU; the graph's destination-vertex range is split by the
reference partitioner (strong scaling: total work fixed), vertex values exchanged every iteration.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

# OpenMP placement of the CPU legs (oracle): spread threads over all cores / NUMA nodes, set before libgomp is loaded.
# ONLY in a process that runs a CPU leg alone (N = 1, or the reference arm where rank 0 works and the others exit): with
# OMP_PROC_BIND set, libgomp pins the MAIN thread to the first place the moment torch loads it — in every rank.  At N > 1
# that put the kernel-enqueuing threads of all ranks on CPU 0, where they time-sliced against each other's spinning
# cudaStreamSynchronize: iterations of 2 ms measured as 4-5 ms (profiles/r02c_bench_n4_* vs r02_trace_exchange_n4.txt).
_AFFINITY0 = os.sched_getaffinity(0) if hasattr(os, "sched_getaffinity") else None
_REFERENCE_ARM = "--impl=reference" in sys.argv or any(a == "--impl" and b == "reference" for a, b in zip(sys.argv, sys.argv[1:]))
_CPU_LEG_PROCESS = int(os.environ.get("WORLD_SIZE", "1")) == 1 or _REFERENCE_ARM
if _CPU_LEG_PROCESS:
    os.environ.setdefault("OMP_PROC_BIND", "spread")
    os.environ.setdefault("OMP_PLACES", "cores")

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

ITERS_PER_STEP = 10
SEED = 27


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--scale", type=int, default=27, help="RMAT scale (27 = BASELINE config; smaller only for debugging)")
    ap.add_argument("--edge-factor", type=int, default=16)
    ap.add_argument("--exchange", default="auto", choices=["auto", "nccl", "p2p"],
                    help="auto = p2p: packed balanced all-gather in three kernels (pack+push, barrier, chunk pull over NVLink)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-ref-gpu", action="store_true")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--reference-split", action="store_true",
                    help="N > 1: work on the reference's greedy edge-balanced split instead of the cost-balanced one")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the PageRank values the last timed step computed (what a caller of "
                         "the timed path reads back; the reference arm: its sampled vertices) to DIR/pagerank_values.npy "
                         "and their vertex ids to DIR/vertex_ids.npy")
    return ap.parse_args()


DUMP_MAX_VERTICES = 4 << 20  # 4 B value + 8 B id each: 48 MiB at most


def dump_outputs(path, values, vid=None):
    """values[i] (float32) belongs to vertex vid[i] (default: i), stored as float64 ids (exact below 2^53).  Beyond
    DUMP_MAX_VERTICES, a fixed, seeded sample of the positions is written (sorted; identical from run to run), so that two
    builds run with the same arguments can be compared output for output."""
    total = len(values)
    vid = np.arange(total, dtype=np.int64) if vid is None else np.asarray(vid)
    if total > DUMP_MAX_VERTICES:
        keep = np.unique(np.random.default_rng(SEED).integers(0, total, DUMP_MAX_VERTICES))
        values, vid = values[keep], vid[keep]
    os.makedirs(path, exist_ok=True)
    np.save(os.path.join(path, "pagerank_values.npy"), np.ascontiguousarray(values, np.float32))
    np.save(os.path.join(path, "vertex_ids.npy"), vid.astype(np.float64))
    return {"dir": path, "vertices_written": int(len(values)), "vertices_computed": int(total)}


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        try:
            p = json.load(open(path))
            return float(p["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:  # noqa: BLE001
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.rows, self.proc, self.index = [], None, index

    def start(self, wait_s=8.0):
        """Started BEFORE the warm-up (B200_PROFILING.md: "start before, kill after"): nvidia-smi's own start-up attaches to
        every GPU of the box and stalls their launch queues for tens of ms — inside a 60 ms multi-GPU timed region that doubled
        the measured iteration time (profiles/r02c_bench_n4_rmat27_nccl_barrier.json vs r02_trace_exchange_n4.txt)."""
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
            t0 = time.time()
            while not self.rows and time.time() - t0 < wait_s and self.proc.poll() is None:
                time.sleep(0.01)  # first row printed = start-up over
        except Exception:  # noqa: BLE001
            self.proc = None

    def mark(self):
        """Index of the next sample: brackets the timed region."""
        return len(self.rows)

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self, lo=0, hi=None):
        """Summary of the samples taken inside [lo, hi) (marks); a timed region shorter than the sampling period falls back
        to every sample since the start of the warm-up (the same load) and says so."""
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:  # noqa: BLE001
            self.proc.kill()
        hi = len(self.rows) if hi is None else hi
        rows, window = self.rows[lo:hi], "timed region"
        if not rows:
            rows, window = self.rows[:max(hi, 1)], "warm-up + timed region (timed region shorter than the 100 ms sampling period)"
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for k, n in enumerate(names):
                if f[3 + k].lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "window": window}


def dist_env():
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    return rank, world, local


def numa_nodes():
    try:
        return len([d for d in os.listdir("/sys/devices/system/node") if d.startswith("node") and d[4:].isdigit()])
    except OSError:
        return None


def oracle_sample(scale, nv, ne, frac_log2, must_cover=(), block_shift=14, seed_sel=12345):
    """A bounded sample of the workload built by the ORACLE's own generator (nothing of the product): destination
    blocks of 2^block_shift consecutive vertices chosen pseudo-randomly (1 in 2^frac_log2 — the representative part,
    identical for every caller) plus the blocks containing every id in must_cover (partition boundaries, hubs).
    Returns (blk, deg, description, blk_random) where blk_random is the representative part alone."""
    import oracle as O
    block_shift = min(block_shift, max(scale - 6, 0))
    n_blocks = ((nv - 1) >> block_shift) + 1
    rng = np.random.default_rng(seed_sel)
    rnd = rng.integers(0, 1 << frac_log2, n_blocks) == 0
    sel = rnd.astype(np.uint8)
    for v in must_cover:
        if 0 <= v < nv:
            sel[int(v) >> block_shift] = 1
    blk = O.rmat_blocks(scale, nv, ne, SEED, block_shift, sel, want_deg=True)
    blk["desc"] = "%d destination blocks of %d vertices (%d vertices, %d of %d edges), oracle generator" % (
        int(sel.sum()), 1 << block_shift, len(blk["vid"]), len(blk["src"]), ne)
    # the representative part: keep the vertices whose block was drawn at random
    keep_v = rnd[blk["vid"].astype(np.int64) >> block_shift]
    if keep_v.all():
        sub = blk
    else:
        ends = blk["row_end"].astype(np.int64)
        begins = np.concatenate([[0], ends[:-1]])
        cnt = (ends - begins)[keep_v]
        keep_e = np.repeat(keep_v, ends - begins)
        sub = dict(vid=blk["vid"][keep_v], row_end=np.cumsum(cnt, dtype=np.uint64), src=np.ascontiguousarray(blk["src"][keep_e]),
                   deg=blk["deg"])
    sub["desc"] = "%d pseudo-random destination blocks of %d vertices (1 in %d; %d vertices, %d of %d edges), oracle generator" % (
        int(rnd.sum()), 1 << block_shift, 1 << frac_log2, len(sub["vid"]), len(sub["src"]), ne)
    return blk, blk["deg"], blk["desc"], sub


def time_oracle_sample(nv, blk, deg, x_old, budget_s, min_runs=3, max_runs=200):
    """Oracle PageRank iterations over the sample on all host cores; returns (MTEPS, cores, per-run seconds)."""
    import oracle as O
    out = np.empty(len(blk["vid"]), np.float32)
    O.pagerank_iter_compact(nv, blk, deg, x_old, out=out)  # warm-up (page faults of `out`, thread pool)
    times, t_all = [], time.perf_counter()
    while len(times) < min_runs or (time.perf_counter() - t_all < budget_s and len(times) < max_runs):
        t0 = time.perf_counter()
        O.pagerank_iter_compact(nv, blk, deg, x_old, out=out)
        times.append(time.perf_counter() - t0)
    return len(blk["src"]) / float(np.median(times)) / 1e6, O.num_threads(), times


def main():
    args = parse_args()
    rank, world, local = dist_env()
    if world != args.gpus and world > 1:
        args.gpus = world
    scale = args.scale
    nv, ne = 1 << scale, args.edge_factor << scale
    workload = "pagerank_pull_rmat%d" % scale
    config = {"workload": workload, "nv": nv, "ne": ne, "iters_per_step": ITERS_PER_STEP, "seed": SEED,
              "rmat": "a,b,c,d=.57,.19,.19,.05 edge_factor %d, duplicates and self-loops kept" % args.edge_factor,
              "l2_policy": "inputs larger than L2 (CSC slice %.1f GB + %.0f MB value replica per GPU vs 126 MB L2)" % (
                  (4 * ne + 8 * nv) / args.gpus / 1e9, 4 * nv / 1e6),
              "parallelism": "dst-range partitions x%d (%s)" % (args.gpus, "reference greedy edge-balanced split" if (
                  args.gpus == 1 or args.reference_split) else "contiguous ranges cut by estimated sweep cost — cfg.balanced_split; "
                  "luxb_partition_bounds still reports the reference's greedy edge-balanced split")}

    if args.impl == "reference":
        if rank != 0:
            return 0
        # The reference has no CPU compute path and cannot be built (Legion missing, SURVEY §8c): this arm times the
        # oracle port on all host cores.  Input: the ORACLE's own generator (nothing of the product is loaded here);
        # a step = ITERS_PER_STEP PageRank iterations over a bounded, representative sample of the destination vertices.
        import oracle as O
        O.set_num_threads(os.cpu_count() or 1)  # torch.distributed.run exports OMP_NUM_THREADS=1 to every rank
        t0 = time.perf_counter()
        _, deg, _, blk = oracle_sample(scale, nv, ne, frac_log2=4)
        desc = blk["desc"]
        x0 = O.pagerank_init(deg)
        t_gen = time.perf_counter() - t0
        out = np.empty(len(blk["vid"]), np.float32)
        edges = len(blk["src"])

        def step():
            t = time.perf_counter()
            for _ in range(ITERS_PER_STEP):
                O.pagerank_iter_compact(nv, blk, deg, x0, out=out)
            return time.perf_counter() - t

        for _ in range(args.warmup):
            step()
        times = [step() for _ in range(args.steps)]
        dumped = dump_outputs(args.dump_outputs, out, blk["vid"]) if args.dump_outputs else None
        total = float(np.sum(times))
        mteps = edges * ITERS_PER_STEP * args.steps / total / 1e6
        sample = "%d iterations per step over %s" % (ITERS_PER_STEP, desc)
        line = {"impl": "reference", "metric": "MTEPS", "value": mteps, "unit": "MTEPS", "n_gpus": args.gpus,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total / args.steps, "higher_is_better": True,
                "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config,
                "cpu_baseline": {"value": mteps, "unit": "MTEPS", "cores": O.num_threads(), "kind": "port", "sample": sample,
                                 "numa_nodes": numa_nodes(), "omp": {k: os.environ.get(k) for k in ("OMP_PROC_BIND", "OMP_PLACES")},
                                 "per_step_seconds": times},
                "e2e": {"value": mteps, "unit": "MTEPS", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0, "input_seconds": t_gen,
                "note": "reference has no CPU compute path and needs Legion (SURVEY §8c): the oracle port is timed; "
                        "input generated by the oracle itself (libluxb is not loaded in this arm)"}
        if dumped:
            line["dump_outputs"] = dumped
        print(json.dumps(line))
        return 0

    import lux_b200 as L

    # ------------------------------------------------------------------------------------------------ ours
    import torch
    if world > 1 and _AFFINITY0 is not None:
        os.sched_setaffinity(0, _AFFINITY0)  # whatever the environment said: the enqueuing thread of a rank is never pinned
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    if args.exchange == "auto":
        args.exchange = "p2p"
    exchange = {"p2p": L.EXCHANGE_P2P, "nccl": L.EXCHANGE_NCCL}[args.exchange]
    t_build0 = time.perf_counter()
    g = L.LuxGraph.from_rmat(scale, nv, ne, SEED, rank=rank, nranks=world, device=local, exchange=exchange,
                             balanced=not args.reference_split)
    g.comm_init_torch()
    g.init()
    if world > 1 and exchange != L.EXCHANGE_NCCL:
        if not g.p2p_connect_torch():  # CUDA IPC unavailable on some rank: every rank degrades to the NCCL exchange
            args.exchange = "nccl (p2p import failed)"
    t_build = time.perf_counter() - t_build0
    view = g.device_view()
    n_part = (view.row_right - view.row_left + 1) & 0xFFFFFFFF
    e_part = view.local_edges

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
            torch.cuda.synchronize()

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()  # before the warm-up: its start-up must not fall into the timed region
    barrier()
    for _ in range(args.warmup):
        g.iterate(ITERS_PER_STEP)

    # ---- device-resident timed region: exactly K steps ----
    g.enable_kernel_timing(True)
    s0 = g.stats()
    barrier()
    m0 = sampler.mark()
    w0 = time.perf_counter()
    for _ in range(args.steps):
        g.iterate(ITERS_PER_STEP)
    barrier()
    w1 = time.perf_counter()
    m1 = sampler.mark()
    s1 = g.stats()
    clocks = sampler.stop(m0, m1) if rank == 0 else None
    g.enable_kernel_timing(False)
    dev_s = s1["loop_seconds"] - s0["loop_seconds"]
    kern_s = s1["dominant_kernel_seconds"] - s0["dominant_kernel_seconds"]
    kern_n = s1["dominant_kernel_launches"] - s0["dominant_kernel_launches"]
    launches = s1["kernel_launches"] - s0["kernel_launches"]
    t = torch.tensor([dev_s, w1 - w0, kern_s / max(kern_n, 1), float(launches)], dtype=torch.float64, device="cuda")
    tsum = t.clone()
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(tsum, op=dist.ReduceOp.SUM)
    dev_s_max, wall_s_max, kern_avg_max = float(t[0]), float(t[1]), float(t[2])
    total_launches = int(tsum[3])
    edges_total = ne * ITERS_PER_STEP * args.steps
    value = edges_total / dev_s_max / 1e6

    dumped = None
    if args.dump_outputs:
        x_last = g.values()  # collective on several ranks
        if rank == 0:
            dumped = dump_outputs(args.dump_outputs, x_last)
        del x_last

    # ---- end to end through the C ABI with host buffers (pinned): every rank moves ITS partition's values over PCIe
    # (luxb_set_local_values: H2D of the slice + device-side exchange; luxb_get_local_values: D2H of the slice), like
    # the per-GPU tasks of the reference touch only their own region.  Together the ranks move nv values each way. ----
    e2e = None
    if not args.no_e2e:
        x_host = torch.empty(max(n_part, 1), dtype=torch.float32).pin_memory()
        y_host = torch.empty(max(n_part, 1), dtype=torch.float32).pin_memory()
        x_np, y_np = x_host.numpy()[:n_part], y_host.numpy()[:n_part]
        g.local_values(out=x_np)
        barrier()
        for _ in range(1):
            g.set_local_values(x_np); g.iterate(ITERS_PER_STEP); g.local_values(out=y_np)
        barrier()
        e0 = time.perf_counter()
        for _ in range(args.steps):
            g.set_local_values(x_np)
            g.iterate(ITERS_PER_STEP)
            g.local_values(out=y_np)
        barrier()
        e1 = time.perf_counter()
        te = torch.tensor([e1 - e0], dtype=torch.float64, device="cuda")
        if dist is not None:
            dist.all_reduce(te, op=dist.ReduceOp.MAX)
        e2e = {"value": edges_total / float(te[0]) / 1e6, "unit": "MTEPS", "h2d_bytes_per_step": 4 * nv,
               "d2h_bytes_per_step": 4 * nv, "ms_per_step": 1e3 * float(te[0]) / args.steps,
               "what": "per rank: luxb_set_local_values(pinned host slice) + luxb_iterate(%d) + luxb_get_local_values(pinned host "
                       "slice) per step; bytes are summed over the ranks; graph structure resident (the reference's timed region "
                       "also excludes load/init, pagerank.cc:108-116)" % ITERS_PER_STEP}

    # ---- roofline of the dominant kernel(s) (this rank's partition): one "launch" = one whole-partition sweep ----
    st_now = g.stats()
    if st_now["panel_edges"]:
        sweep_kernel = ("seg_tile_kernel<panel: %d hubs x %d hot-source blocks in shared memory, %.1f%% of the edges> + panel fix-up + "
                        "seg_tile_kernel<main, L1 gathers>" % (st_now["panel_hubs"], st_now["panel_blocks"], 100.0 * st_now["panel_edges"] / max(e_part, 1)))
    else:
        sweep_kernel = "seg_tile_kernel<main, L1 gathers>"
    peak, peak_src = load_peaks()
    algo_bytes = 8 * e_part + 16 * n_part  # SURVEY §8(d): 4 B src id + 4 B gathered value per edge; 8+4+4 per vertex
    achieved = algo_bytes / max(kern_avg_max, 1e-12) / 1e9
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": None, "kernel": sweep_kernel, "avg_launch_ms": 1e3 * kern_avg_max,
                "algorithmic_bytes_per_launch": algo_bytes, "peak_source": peak_src,
                "note": "traffic: see profiles/ (ncu dram__bytes_read.sum + dram__bytes_write.sum)"}
    prof = os.path.join(ROOT, "profiles", "r02_traffic.json")
    if os.path.exists(prof) and world == 1:  # ncu dram__bytes_read.sum + dram__bytes_write.sum of the 1-GPU sweep kernels
        try:
            roofline["traffic"] = json.load(open(prof)).get(workload)
        except Exception:  # noqa: BLE001
            pass

    # ---- the reference's OWN CUDA kernels on the same box (oracle/_ref/libref_pagerank.so: pagerank_gpu.cu compiled
    # unmodified behind a Legion shim, zero-copy regions emulated with mapped pinned memory).  Its init does a host
    # std::sort of all edges (pagerank_gpu.cu:229-242), minutes at RMAT-27, so both engines are timed on RMAT-24. ----
    ref_gpu = None
    if rank == 0 and world == 1 and not args.no_ref_gpu:
        try:
            from oracle import refrun as R
            if R.available("pagerank"):
                sc = min(scale, 24)
                nv2, ne2 = 1 << sc, args.edge_factor << sc
                with L.LuxGraph.from_rmat(sc, nv2, ne2, SEED, device=local) as g2:
                    re2, src2 = g2.local_csc()
                    g2.init()
                    g2.iterate(3)
                    a0 = g2.stats()
                    g2.iterate(ITERS_PER_STEP)
                    a1 = g2.stats()
                    ours_ms = 1e3 * (a1["loop_seconds"] - a0["loop_seconds"]) / ITERS_PER_STEP
                _, ref_ms = R.pagerank(re2, src2, ITERS_PER_STEP)
                ref_ms /= ITERS_PER_STEP
                ref_gpu = {"workload": "pagerank_pull_rmat%d" % sc, "reference_MTEPS": ne2 / ref_ms / 1e3,
                           "ours_MTEPS_same_graph": ne2 / ours_ms / 1e3, "reference_ms_per_iter": ref_ms,
                           "ours_ms_per_iter": ours_ms, "how": "reference task bodies + kernels replayed (oracle/ref_replay), 1 partition"}
        except Exception as e:  # noqa: BLE001
            ref_gpu = {"unavailable": repr(e)[:200]}

    # ---- parity at this N (after the timed region): the device's state x_k, ONE more device iteration, and on rank 0
    # one ORACLE iteration from x_k over a sample of destination blocks generated by the oracle itself — pseudo-random
    # blocks plus the blocks around every partition boundary and vertex 0 (hubs), so every rank's slice and therefore
    # the exchange is covered.  The same sample feeds the CPU baseline at N = 1. ----
    parity, cpu_base = None, None
    if not args.no_parity:
        x_k = g.values()   # collective on several ranks: completes the natural-order replica (exchanged packed otherwise)
        g.iterate(1)
        x_k1 = g.values()
        if rank == 0:
            import oracle as O
            O.set_num_threads(os.cpu_count() or 1)  # torch.distributed.run exports OMP_NUM_THREADS=1 to every rank
            b = g.work_bounds()
            cover = [0, nv - 1]
            for p in range(world):
                cover += [int(b["row_left"][p]), int(b["row_right"][p]) & 0xFFFFFFFF]
            blk, deg_o, desc, blk_rnd = oracle_sample(scale, nv, ne, frac_log2=4, must_cover=cover)
            ref = O.pagerank_iter_compact(nv, blk, deg_o, x_k)
            got = x_k1[blk["vid"]]
            rel = np.abs(got.astype(np.float64) - ref.astype(np.float64)) / np.maximum(np.abs(ref.astype(np.float64)), 1e-300)
            deg_dev_ok = None
            if world == 1:
                deg_dev_ok = bool(np.array_equal(g.out_degree(), deg_o))
            parity = {"max_rel_err": float(rel.max()), "tolerance": 1e-6, "ok": bool(rel.max() <= 1e-6),
                      "checked_vertices": int(len(ref)), "checked_edges": int(len(blk["src"])), "sample": desc,
                      "partitions_covered": world, "device_out_degrees_equal_oracle": deg_dev_ok,
                      "what": "device x_k -> one device iteration vs one oracle iteration (fp64 sums) on the sample"}
            if world == 1 and not args.no_cpu_baseline:
                # x_k came back from the device through one host thread (all its pages on one NUMA node): time the oracle
                # on a copy whose pages were first touched by the OpenMP threads, like the reference arm's x0
                x_par = O.pagerank_init(deg_o)
                np.copyto(x_par, x_k)
                mteps, cores, times = time_oracle_sample(nv, blk_rnd, deg_o, x_par, budget_s=12.0)
                cpu_base = {"value": mteps, "unit": "MTEPS", "cores": cores, "kind": "port", "numa_nodes": numa_nodes(),
                            "sample": "1 PageRank iteration over %s (the reference arm's sample), median of %d runs" % (
                                blk_rnd["desc"], len(times))}
    g.close()

    if rank == 0:
        line = {"metric": "MTEPS", "value": value, "unit": "MTEPS", "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": 1e3 * dev_s_max / args.steps, "higher_is_better": True,
                "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config,
                "e2e": e2e, "gpu_launches": total_launches, "roofline": roofline, "cpu_baseline": cpu_base,
                "parity": parity, "reference_gpu_replay": ref_gpu, "clocks": clocks, "wall_ms_per_step": 1e3 * wall_s_max / args.steps, "build_seconds": t_build,
                "exchange": args.exchange if world > 1 else "none",
                "roofline_whole_step": {"algorithmic_GBps_per_gpu": (8 * ne + 16 * nv) * ITERS_PER_STEP * args.steps
                                        / world / dev_s_max / 1e9, "frac": (8 * ne + 16 * nv) * ITERS_PER_STEP
                                        * args.steps / world / dev_s_max / 1e9 / peak}}
        if dumped:
            line["dump_outputs"] = dumped
        print(json.dumps(line))
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
