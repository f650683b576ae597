#!/usr/bin/env python3
"""bench.py — primitive expansions/s of the batched lattice planner (BASELINE.json metric).

  python bench.py --gpus N --steps K --warmup W            this repo's CUDA path (one process per GPU)
  python bench.py --impl reference --gpus N --steps K ...   the reference's CPU implementation on host cores: its own
                                                            sources (oracle/_ref, stand-in Eigen/Boost headers) when
                                                            that binary is present, else the oracle port
  --workload c2 (default) | c5        --queries Q (default 65536)
  --dump-outputs DIR                  the last timed step's result records and action rows as DIR/<name>.npy (dump_outputs)

Workloads (SURVEY.md §8d, mpl_ros_b200/workloads.py):
  c2  BASELINE configs[1] scaled to the north-star batch: levine-256 (levine.bag upsampled 2x, cropped, placed in a 256^3
      int8 grid), |U| = 27 acceleration controls, dt = 1, v_max = 2, a_max = 1, tol_pos = 0.5; ONE list of 65 536
      (start, goal) pairs, RandomState(0), unreachable pairs kept.  The list is sharded over the N ranks (query i ->
      rank i mod N: strong scaling).  The literal configs[1] batch (the first 1024 queries of the list, one GPU) is
      measured in the same run and reported under config.batch1024.
  c5  BASELINE configs[4]: synthetic 1024^3 box map, |U| = 125 jerk controls, dt = 0.5, v_max = 3, a_max = 2,
      max_num = 50 000, 65 536 pairs RandomState(2) with L-inf distance in [3 m, 30 m].
A "step" is one pass of the whole list through the planner: every rank plans its stripe, rank 0 gathers the result
records and action rows (the one data-path collective).  Unit of work: one primitive expansion = one (popped state, u)
pair entering env_map.h:155.

`value`   : device-resident stripes (ShardedBatchPlanner.plan_stripe_device -> mplb_plan_stripe_gather_device: the search
            kernel + the ncclSend/ncclRecv gather inside libmplb), CUDA events on the launch stream, max over ranks.
`e2e`     : the public host-buffer call (ShardedBatchPlanner.plan_batch -> mplb_plan_batch_sharded) with the full list in
            pinned host memory on every rank: H2D of the stripe's starts/goals, the gather and D2H of results + action
            rows inside the timed region.
`roofline`: ALGORITHMIC bytes per primitive expansion (SURVEY.md §8d formula, recomputed from the kernel's own
            counters) x expansions per launch / launch duration, against MEASURED_PEAKS.json hbm_gbs.
`cpu_baseline`: the reference's CPU path on this box's host cores, bounded sample (dynamic work queue over the sample,
            longest plans first, threads pinned): oracle/_ref ("reference") when present, else the oracle port ("port").
"""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

MAX_SEG = 64


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "measured"
    return 6650.0, "fallback"


def workload(name):
    from mpl_ros_b200 import workloads as W
    if name == "c2":
        return dict(spec=W.C2, tag="levine256_U27_acc", make_map=W.c2_map, make_queries=W.c2_queries,
                    map_note="levine-256 (256^3 int8, 16 MiB; kernel reads 2 MiB of occupancy bit-bricks)",
                    b_state=56.0, b_succ=72.0, kernel="astar_batch_kernel<3,2,1,0>", cpu_sample=1024, cpu_threads=None,
                    mem_fraction=None)
    return dict(spec=W.C5, tag="boxes1024_U125_jrk", make_map=W.c5_map, make_queries=W.c5_queries,
                map_note="synthetic boxes 1024^3 int8 (1 GiB; kernel reads 128 MiB of occupancy bit-bricks)",
                b_state=80.0, b_succ=96.0, kernel="astar_batch_kernel<3,3,4,0>", cpu_sample=16, cpu_threads=16,
                mem_fraction=0.85)


SEARCH_UNITS = ("mplb.cu", "mplb_device.cuh", "mplb_search.cuh", "mplb_trig.cuh")  # the search kernel and its launch code


def src_sha():
    """Hash of the sources of the search kernel and of the host code that launches it: profiles/traffic.json entries are
    only trusted for the code they were captured on (the LPA* and TrajSolver units are separate translation units that the
    bench launch never touches)."""
    h = hashlib.sha256()
    d = os.path.join(ROOT, "mpl_ros_b200", "csrc")
    for f in SEARCH_UNITS:
        h.update(open(os.path.join(d, f), "rb").read())
    return h.hexdigest()[:16]


def b_alg(res, nU, wl):
    """SURVEY.md §8(d): B_alg = B_state/|U| + S_mean*1 + p_valid*(B_succ + B_probe)."""
    prims = float(res["n_prims"].sum())
    s_mean = float(res["n_samples"].sum()) / prims
    p_valid = float(res["n_valid"].sum()) / prims
    return wl["b_state"] / nU + s_mean + p_valid * (wl["b_succ"] + 16.0), s_mean, p_valid


DUMP_BYTES = 64 * 10 ** 6


def dump_outputs(d, res, acts):
    """Writes what the timed path hands its caller after the last timed step, one row per query in global order: every
    field of the result records as float64 (the 64-bit key hashes as two exact 32-bit halves, `_lo` and `_hi`; the
    infinite cost of a plan that found no path as -1, which no path costs; device_ms, a timing, is left out) and the action
    rows as float32 (-1 pads a plan's unused rows).  Every value is finite.  Above DUMP_BYTES, a fixed RandomState(0)
    sample of the rows; query_index.npy names the rows either way."""
    cols = {}
    for f in res.dtype.names:
        if f == "device_ms":
            continue
        if res[f].dtype == np.uint64:
            cols[f + "_lo"], cols[f + "_hi"] = res[f] & 0xFFFFFFFF, res[f] >> 32
        else:
            cols[f] = res[f]
    cols["cost"] = np.where(np.isinf(cols["cost"]), -1.0, cols["cost"])
    n = len(res)
    row_bytes = 8 * (len(cols) + 1) + 4 * acts.shape[1]
    idx = np.arange(n)
    room = DUMP_BYTES - 128 * (len(cols) + 2)  # less one .npy header per file
    if n * row_bytes > room:
        idx = np.sort(np.random.RandomState(0).choice(n, room // row_bytes, replace=False))
    out = {name: v[idx].astype(np.float64) for name, v in cols.items()}
    out["query_index"], out["actions"] = idx.astype(np.float64), acts[idx].astype(np.float32)
    bad = [name for name, v in out.items() if not np.isfinite(v).all()]
    assert not bad, "non-finite outputs: %s" % bad
    os.makedirs(d, exist_ok=True)
    for name, v in out.items():
        np.save(os.path.join(d, name + ".npy"), v)


def lpt_order(m, S, G):
    """Longest-plans-first processing order for the CPU queue (scheduling only): queries whose goal lies in another
    free-space component exhaust the start's component, then larger L-inf distance first — the same hint the GPU path
    computes with its own label kernels."""
    try:
        from scipy import ndimage
    except Exception:
        return None
    nd = tuple(int(x) for x in m.dim[::-1])
    if int(np.prod(nd)) > (1 << 26):
        return None
    lab, _ = ndimage.label(m.data.reshape(nd) != 100)
    size = np.bincount(lab.ravel())

    def cell(P):
        c = np.floor((P - m.origin) / m.res).astype(np.int64)
        c = np.clip(c, 0, m.dim.astype(np.int64) - 1)
        return lab[c[:, 2], c[:, 1], c[:, 0]] if m.ndim == 3 else lab[c[:, 1], c[:, 0]]
    ls, lg = cell(S), cell(G)
    dist = np.abs(S - G).max(axis=1)
    key = np.where((ls != lg) & (ls > 0), 1e9 + size[ls], dist)
    return np.argsort(-key, kind="stable").astype(np.int32)


class ClockSampler:
    """nvidia-smi clocks/throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap,timestamp")

    def __init__(self, gpu):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(gpu), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                       "-lms", "100"], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self, t0=None, t1=None):
        """t0/t1: wall-clock window (time.time()) of the timed region; samples outside it are dropped when at least
        three fall inside (the sampler is started before the warm-up because nvidia-smi takes ~0.5 s to start)."""
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.p.terminate()
        self.p.wait()
        self.f.flush()
        rows = [r.split(", ") for r in open(self.f.name).read().strip().splitlines() if r.strip()]
        os.unlink(self.f.name)
        rows = [r for r in rows if len(r) >= 10]
        window = "timed region"
        if t0 is not None:
            import datetime
            inside = []
            for r in rows:
                try:
                    ts = datetime.datetime.strptime(r[9].strip(), "%Y/%m/%d %H:%M:%S.%f").timestamp()
                except ValueError:
                    continue
                if t0 - 0.05 <= ts <= t1 + 0.05:
                    inside.append(r)
            if len(inside) >= 3:
                rows = inside
            else:
                window = "warm-up + timed region (fewer than 3 samples fell inside the timed region)"
        sm = [float(r[1]) for r in rows if len(r) >= 9]
        reasons = set()
        for r in rows:
            if len(r) < 9:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                if v.strip().lower() == "active":
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": float(rows[0][2]) if rows else None,
                "samples": len(sm), "window": window, "reasons": sorted(reasons)}


KIND_NOTE = {"reference": "the reference's own planner sources (oracle/_ref: stand-in Eigen/Boost headers, see oracle/shim)",
             "port": "oracle port (oracle/_ref absent)"}


def cpu_planners(m, U, wl):
    """{'port': planner, 'reference': planner or absent}; both expose plan_batch(s, g, nthreads, order, pin, want_busy)."""
    import oracle
    params = wl["spec"]["params"]
    out = {}
    om = oracle.OracleMap(m.origin, m.dim, m.data, m.res)
    om.free_unknown()
    op = oracle.OraclePlanner(3)
    op.set_map(om)
    for k, v in params.items():
        op.set_param(k, v)
    op.set_controls(U)
    op._keep = om

    class _Port:
        def plan_batch(self, s, g, **kw):
            r = op.plan_batch(s, g, want_busy=True, **kw)
            return r[0], r[2]
    out["port"] = _Port()
    try:
        from oracle import ref
        if ref.available():
            rm = ref.RefMap(m.origin, m.dim, m.data, m.res)
            rm.free_unknown()
            rp = ref.RefPlanner(3)
            rp.set_map(rm)
            for k, v in params.items():
                rp.set_param(k, v)
            rp.set_controls(U)
            rp._keep = rm

            class _Ref:
                def plan_batch(self, s, g, **kw):
                    return rp.plan_batch(s, g, want_busy=True, **kw)
            out["reference"] = _Ref()
    except Exception as e:  # a broken checker build must not take the bench line down: the port always exists
        out["reference_error"] = repr(e)[:200]
    return out


def cpu_sample_queries(S, G, control, n):
    import oracle
    so, go = oracle.make_waypoints(n), oracle.make_waypoints(n)
    so["pos"], go["pos"], so["control"], go["control"] = S[:n], G[:n], control, control
    return so, go


def time_cpu(pl, so, go, threads, order):
    t0 = time.perf_counter()
    res, busy = pl.plan_batch(so, go, nthreads=threads, order=order, pin=True)
    dt = time.perf_counter() - t0
    return res, dt, float(busy.sum() / (dt * threads))


def run_reference(args):
    """The reference's CPU implementation of the path, all host threads, a bounded sample of the same workload per step."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    wl = workload(args.workload)
    from mpl_ros_b200 import workloads as W
    m = wl["make_map"]()
    U = W.controls(wl["spec"])
    n_s = args.cpu_sample or wl["cpu_sample"]
    S, G = wl["make_queries"](m, n_s)
    pls = cpu_planners(m, U, wl)
    kind = "reference" if "reference" in pls else "port"
    pl = pls[kind]
    cores = os.cpu_count() or 1
    threads = min(cores, wl["cpu_threads"] or cores, n_s)
    so, go = cpu_sample_queries(S, G, wl["spec"]["control"], n_s)
    order = lpt_order(m, S, G)
    for _ in range(args.warmup):
        pl.plan_batch(so[:min(threads, n_s)], go[:min(threads, n_s)], nthreads=threads, pin=True)
    t0 = time.perf_counter()
    prims, util, ms_all = 0, [], []
    for _ in range(args.steps):
        res, dt, u = time_cpu(pl, so, go, threads, order)
        prims += int(res["n_prims"].sum())
        util.append(u)
        ms_all.append(res["device_ms"])
    dt = time.perf_counter() - t0
    v = prims / dt
    ms_all = np.concatenate(ms_all)
    sample = "first %d of the %d queries per step (bounded sample), atomic work queue, longest plans first, threads pinned" % (
        n_s, wl["spec"]["n_queries"])
    line = {"impl": "reference", "metric": "primitive_expansions_per_sec", "value": v, "unit": "prim_exp/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": "%s_batch%d" % (wl["tag"], wl["spec"]["n_queries"]), "step": sample,
                       "ms_per_plan_p50": float(np.percentile(ms_all, 50)), "ms_per_plan_p95": float(np.percentile(ms_all, 95))},
            "cpu_baseline": {"value": v, "unit": "prim_exp/s", "cores": threads, "kind": kind, "what": KIND_NOTE[kind],
                             "sample": sample, "thread_utilisation": float(np.mean(util))},
            "e2e": {"value": v, "unit": "prim_exp/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="mplb", choices=["mplb", "reference"])
    ap.add_argument("--workload", default="c2", choices=["c2", "c5"])
    ap.add_argument("--queries", type=int, default=0, help="length of the global query list (default: the workload's 65536)")
    ap.add_argument("--cpu-sample", type=int, default=0, help="queries in the CPU-baseline sample (default per workload)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-batch1024", action="store_true")
    ap.add_argument("--pipeline", action="store_true",
                    help="N = 1 only: two planners alternate so that the drain of one launch overlaps the start of the next "
                         "(mplb_plan_stripe_begin / _end); off by default — with N > 1 the NCCL gather kernel cannot get SM room "
                         "beside a persistent search kernel that fills the GPU, so the overlap does not materialise there")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the result records and action rows of the last one as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.warmup < 3:
        args.warmup = 3
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import mpl_ros_b200 as mp
    from mpl_ros_b200 import _lib, workloads as W
    from mpl_ros_b200 import dist as mdist

    wl = workload(args.workload)
    spec = wl["spec"]
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: libmplb has no CPU path")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist = None
    # stdout carries the one JSON line: NCCL's own log (NCCL_DEBUG as the caller set it; libmplb's communicator initialises
    # NCCL at every world size) goes to a file in the temporary directory unless the caller already chose one
    if os.environ.get("NCCL_DEBUG") and not os.environ.get("NCCL_DEBUG_FILE"):
        os.environ["NCCL_DEBUG_FILE"] = os.path.join(tempfile.gettempdir(), "nccl.bench.%h.%p.log")
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)

    # ---- map and the ONE query list: rank 0 builds both; one NCCL broadcast of the grid puts the map in every GPU's
    # HBM (SURVEY.md §8e), one broadcast hands every rank the list it takes its stripe from
    U = W.controls(spec)
    nq = args.queries or spec["n_queries"]
    m = wl["make_map"]() if rank == 0 else None

    def make_planner(o, d, r, mu, first=True):  # mu: the MapUtil that mplb_comm_broadcast_map built on this rank's device
        if first:
            mu.freeUnknown()
        pl = mp.VoxelMapPlanner(False)
        pl.setMapUtil(mu)
        p = spec["params"]
        pl.setVmax(p["v_max"]); pl.setAmax(p["a_max"]); pl.setDt(p["dt"]); pl.setU(U); pl.setTol(p["tol_pos"])
        if "max_num" in p:
            pl.setMaxNum(p["max_num"])
        if wl["mem_fraction"]:
            pl.setMemFraction(wl["mem_fraction"])
        pl._keep = mu
        return pl

    # the two data-path collectives (grid broadcast, result gather) run inside libmplb on its own NCCL communicator;
    # torch.distributed only carries the communicator id, the query list and the timing reductions
    comm = mdist.Comm.from_process_group(dev)
    sp = mdist.ShardedBatchPlanner(make_planner, dev, comm=comm)
    if m is not None:
        sp.set_map(m.origin, m.dim, m.res, m.data)
    else:
        sp.set_map()
    pl = sp.planner
    # --pipeline: a second planner on the same map and communicator; batches alternate between the two, so that the drain of
    # one launch (it ends with its longest plan) overlaps the start of the next
    pipe = bool(args.pipeline) and world == 1 and args.workload == "c2"
    sp2 = None
    if pipe:
        sp2 = mdist.ShardedBatchPlanner(make_planner, dev, comm=comm)
        sp2.planner = make_planner(None, None, None, pl.map_util_, first=False)
    s_all, g_all = mp.waypoints_array(nq), mp.waypoints_array(nq)
    if rank == 0:
        S, G = wl["make_queries"](m, nq)
        W.fill(s_all, g_all, S, G, spec["control"])
    s_all, g_all = sp.broadcast_queries(s_all, g_all)
    idx = mdist.shard_indices(nq, rank, world)
    n_loc = len(idx)
    hs = torch.from_numpy(np.ascontiguousarray(s_all[idx]).view(np.uint8).reshape(n_loc, -1)).pin_memory()
    hg = torch.from_numpy(np.ascontiguousarray(g_all[idx]).view(np.uint8).reshape(n_loc, -1)).pin_memory()
    ds, dg = hs.to(dev), hg.to(dev)
    flush = torch.empty(512 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2
    stream = torch.cuda.current_stream()
    bufs = sp.make_device_buffers(nq, MAX_SEG)

    def step_device():
        return sp.plan_stripe_device(ds, dg, n_loc, bufs, MAX_SEG, stream)

    sps = [sp, sp2] if pipe else [sp]
    pbufs = [bufs] + ([sp2.make_device_buffers(nq, MAX_SEG)] if pipe else [])
    pstreams = [torch.cuda.Stream(device=dev) for _ in sps]

    def run_pipelined(k_steps):
        """k_steps batches, at most one in flight per planner: begin(k), then end(k - 1).  Returns the device time of the
        whole region (events on the default stream around it, the device idle at both ends) and the planner of the last batch."""
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for k in range(k_steps):
            flush.zero_()  # L2 flush between iterations (default stream, concurrent with the batch still draining)
            i = k % len(sps)
            sps[i].begin_stripe_device(ds, dg, n_loc, pbufs[i], MAX_SEG, pstreams[i])
            if k > 0:
                j = (k - 1) % len(sps)
                sps[j].end_stripe_device(pbufs[j])
        last = (k_steps - 1) % len(sps)
        sps[last].end_stripe_device(pbufs[last])
        torch.cuda.synchronize()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1), last

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    clocks = ClockSampler(local)
    if pipe:
        run_pipelined(args.warmup)
        barrier()
        launches0 = _lib.lib().mplb_launch_count()
        t_wall0 = time.time()
        total_ms, last = run_pipelined(args.steps)
        barrier()
        t_wall1 = time.time()
        kernel_ms = [total_ms / args.steps]  # launches overlap: the per-launch share of the timed region
        lastbufs = pbufs[last]
    else:
        for _ in range(args.warmup):
            flush.zero_()
            step_device()
        barrier()
        launches0 = _lib.lib().mplb_launch_count()
        t_wall0 = time.time()
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
        kernel_ms = []
        for k in range(args.steps):
            flush.zero_()  # L2 flush between timed iterations (outside the event pair)
            ev[k][0].record(stream)
            step_device()
            ev[k][1].record(stream)
            kernel_ms.append(pl.last_batch_stats()["kernel_ms"])
        barrier()
        t_wall1 = time.time()
        total_ms = float(sum(a.elapsed_time(b) for a, b in ev))
        lastbufs = bufs
    clk = clocks.stop(t_wall0, t_wall1)
    launches = int(_lib.lib().mplb_launch_count() - launches0)
    res_loc = lastbufs["res"].cpu().numpy().view(_lib.RESULT_DTYPE).reshape(-1)[:n_loc]
    res_all, acts_all = sp.unstripe(lastbufs, nq, MAX_SEG) if rank == 0 else (None, None)
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, res_all, acts_all)

    # ---- e2e through the public host-buffer API (pinned inputs, H2D + D2H + gather inside the timed region)
    s_pin = torch.from_numpy(s_all.view(np.uint8).reshape(nq, -1)).pin_memory().numpy().view(_lib.WAYPOINT_DTYPE).reshape(-1)
    g_pin = torch.from_numpy(g_all.view(np.uint8).reshape(nq, -1)).pin_memory().numpy().view(_lib.WAYPOINT_DTYPE).reshape(-1)
    sp.plan_batch(s_pin, g_pin, MAX_SEG)
    barrier()
    e2e_steps = max(2, min(args.steps, int(30e3 * args.steps / max(total_ms, 1.0))))
    flush_ms = 0.0
    tf0, tf1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    tf0.record(); flush.zero_(); tf1.record(); torch.cuda.synchronize()
    flush_ms = tf0.elapsed_time(tf1)
    barrier()
    t0 = time.perf_counter()
    if pipe:  # the same alternation through the host-buffer calls: begin(k) copies and enqueues, end(k - 1) gathers and copies back
        for k in range(e2e_steps):
            flush.zero_()
            sps[k % 2].begin_batch(s_pin, g_pin, MAX_SEG)
            if k > 0:
                res_h, acts_h = sps[(k - 1) % 2].end_batch()
        res_h, acts_h = sps[(e2e_steps - 1) % 2].end_batch()
        torch.cuda.synchronize()
        flush_ms = 0.0  # the flushes ran concurrently with the batches
    else:
        for _ in range(e2e_steps):
            flush.zero_()
            torch.cuda.synchronize()
            res_h, acts_h = sp.plan_batch(s_pin, g_pin, MAX_SEG)
    barrier()
    e2e_ms = ((time.perf_counter() - t0) * 1e3 - flush_ms * e2e_steps) / e2e_steps
    if rank == 0:
        for f in ("status", "pops", "n_nodes", "pop_hash", "closed_hash", "n_seg"):
            assert np.array_equal(res_h[f], res_all[f]), "host-API results differ from device-API results: " + f

    # ---- secondary, N > 1 only: weak scaling — every rank plans the WHOLE list (65 536 plans per GPU, the launch size of the
    # N = 1 line), no gather; reported beside the strong-scaling headline as config.weak_scaling
    weak_ms = 0.0
    if world > 1 and args.workload == "c2":
        dsa = torch.from_numpy(s_all.view(np.uint8).reshape(nq, -1)).to(dev)
        dga = torch.from_numpy(g_all.view(np.uint8).reshape(nq, -1)).to(dev)
        wres = torch.zeros(nq, _lib.RESULT_DTYPE.itemsize, dtype=torch.uint8, device=dev)
        for _ in range(1):
            pl.plan_batch_device(dsa.data_ptr(), dga.data_ptr(), nq, wres.data_ptr(), 0, 0, 0, stream.cuda_stream)
        barrier()
        w0, w1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        w0.record(stream)
        for _ in range(2):
            pl.plan_batch_device(dsa.data_ptr(), dga.data_ptr(), nq, wres.data_ptr(), 0, 0, 0, stream.cuda_stream)
        w1.record(stream)
        barrier()
        weak_ms = w0.elapsed_time(w1) / 2

    # ---- multi-GPU: max over ranks of the timed region
    tot = np.array([total_ms, e2e_ms, float(np.mean(kernel_ms)), weak_ms])
    if dist is not None:
        t = torch.tensor(tot, dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        total_ms, e2e_ms, kms_max, weak_ms = (float(x) for x in t.cpu().numpy())
    else:
        kms_max = float(np.mean(kernel_ms))
    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return

    prims_all, pops_all = float(res_all["n_prims"].sum()), float(res_all["pops"].sum())
    ms_step = total_ms / args.steps
    value = prims_all / (ms_step * 1e-3)
    e2e_v = prims_all / (e2e_ms * 1e-3)
    peak, peak_kind = load_peaks()
    balg, s_mean, p_valid = b_alg(res_loc, U.shape[0], wl)
    kms = float(np.mean(kernel_ms))
    ach = float(res_loc["n_prims"].sum()) * balg / (kms * 1e-3) / 1e9
    traffic, traffic_note = None, "no ncu capture recorded for this workload"
    prof = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(prof):
        ent = json.load(open(prof)).get(args.workload)
        if ent and ent.get("src_sha") == src_sha() and ent.get("queries_per_launch") == n_loc:
            traffic, traffic_note = ent["dram_bytes_per_launch"], "ncu --set full capture %s of this code and launch size" % ent.get("capture", "")
        elif ent:
            traffic_note = "stale: the recorded capture is of other kernel sources or another launch size"

    dms = res_all["device_ms"]
    # single-plan latency through the public API (what map_planner_node does): a few queries one at a time
    lat = []
    for i in range(min(8, nq)):
        a, b = s_all[i:i + 1].copy(), g_all[i:i + 1].copy()
        t0 = time.perf_counter()
        pl.plan(a, b)
        lat.append((time.perf_counter() - t0) * 1e3)

    ok = res_all["status"] == 0
    cfg = {"workload": "%s_batch%d" % (wl["tag"], nq), "map": wl["map_note"], "U": int(U.shape[0]), "global_batch": nq,
           "parallelism": "one query list sharded over %d rank(s), query i -> rank i mod N; map broadcast + result gather" % world,
           "l2": "flushed between timed iterations (512 MiB memset per step)",
           "pipeline": ("two planners alternate: batch k + 1 is enqueued before batch k is waited for, so the drain of a launch "
                        "overlaps the start of the next; value = units / (device time of the K-step region / K)") if pipe else "off",
           "plans_per_sec": nq / (ms_step * 1e-3),
           "ms_per_plan_p50": float(np.percentile(dms, 50)), "ms_per_plan_p95": float(np.percentile(dms, 95)),
           "ms_per_plan_max": float(dms.max()),
           "ms_per_plan_note": "device time of each plan inside the batch (mplb_result.device_ms), all ranks",
           "single_plan_api_ms_p50": float(np.median(lat)),
           "node_expansions_per_sec": pops_all / (ms_step * 1e-3),
           "success_rate": float(ok.mean()), "unreachable_rate": float((res_all["status"] == 3).mean()),
           "max_expand_rate": float((res_all["status"] == 2).mean()),
           "mean_samples_per_prim": s_mean, "p_valid": p_valid, "e2e_steps": e2e_steps}
    if weak_ms > 0:
        cfg["weak_scaling"] = {"what": "every rank plans the whole %d-query list (the N = 1 launch size), no gather; max over ranks" % nq,
                               "value": world * prims_all / (weak_ms * 1e-3), "unit": "prim_exp/s", "ms_per_step": weak_ms, "steps": 2}
    line = {
        "metric": "primitive_expansions_per_sec", "value": value, "unit": "prim_exp/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": cfg,
        "e2e": {"value": e2e_v, "unit": "prim_exp/s",
                "h2d_bytes_per_step": int(2 * nq * _lib.WAYPOINT_DTYPE.itemsize),
                "d2h_bytes_per_step": int(nq * (_lib.RESULT_DTYPE.itemsize + 4 * MAX_SEG))},
        "gpu_launches": launches,
        "clocks": clk,
        "roofline": {"bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak, "traffic": traffic,
                     "traffic_note": traffic_note, "kernel": wl["kernel"], "alg_bytes_per_prim": balg,
                     "peak_kind": peak_kind + " (burst copy)", "kernel_ms_per_launch": kms,
                     "kernel_ms_per_launch_max_over_ranks": kms_max,
                     "note": "latency/issue-bound search bookkeeping, not HBM-bound: see DESIGN.md roofline section"},
    }

    # ---- the literal configs[1] batch: the first 1024 queries on one GPU (N = 1 only)
    if world == 1 and not args.no_batch1024 and nq >= 1024 and args.workload == "c2":
        nb = 1024
        b = sp.make_device_buffers(nb, MAX_SEG)
        d1s, d1g = ds[:nb].contiguous(), dg[:nb].contiguous()
        for _ in range(3):
            flush.zero_()
            sp.plan_stripe_device(d1s, d1g, nb, b, MAX_SEG, stream)
        torch.cuda.synchronize()
        nst = min(args.steps, 10)
        e1 = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(nst)]
        for k in range(nst):
            flush.zero_()
            e1[k][0].record(stream)
            sp.plan_stripe_device(d1s, d1g, nb, b, MAX_SEG, stream)
            e1[k][1].record(stream)
        torch.cuda.synchronize()
        ms1 = float(np.mean([x.elapsed_time(y) for x, y in e1]))
        r1 = b["res"].cpu().numpy().view(_lib.RESULT_DTYPE).reshape(-1)[:nb]
        cfg["batch1024"] = {"what": "BASELINE configs[1] as literally stated: the first 1024 queries of the list in one launch",
                            "value": float(r1["n_prims"].sum()) / (ms1 * 1e-3), "unit": "prim_exp/s", "ms_per_step": ms1,
                            "steps": nst, "ms_per_plan_p50": float(np.percentile(r1["device_ms"], 50)),
                            "ms_per_plan_p95": float(np.percentile(r1["device_ms"], 95))}

    if not args.no_cpu_baseline:
        n_s = min(args.cpu_sample or wl["cpu_sample"], nq)
        cores = os.cpu_count() or 1
        threads = min(cores, wl["cpu_threads"] or cores, n_s)
        Sq, Gq = s_all["pos"][:n_s], g_all["pos"][:n_s]
        so, go = cpu_sample_queries(Sq, Gq, spec["control"], n_s)
        order = lpt_order(m, Sq, Gq)
        pls = cpu_planners(m, U, wl)
        ro, dt_port, util_port = time_cpu(pls["port"], so, go, threads, order)
        n1 = min(8, n_s)
        r1c, dt_1, _ = time_cpu(pls["port"], so[:n1], go[:n1], 1, None)
        for f in ("status", "pops", "n_nodes", "pop_hash", "closed_hash", "cost"):  # the sample doubles as an in-bench parity check
            a, b2 = ro[f], res_all[f][:n_s]
            assert np.array_equal(a, b2) or f == "cost" and np.array_equal(a[np.isfinite(a)], b2[np.isfinite(b2)]), f
        port_v = float(ro["n_prims"].sum()) / dt_port
        sample = ("first %d of the %d queries, atomic work queue (longest plans first), %d pinned threads; GPU results for "
                  "the same queries checked equal against the oracle port" % (n_s, nq, threads))
        cb = {"value": port_v, "unit": "prim_exp/s", "cores": threads, "host_cores": cores, "kind": "port",
              "thread_utilisation": util_port, "single_core_value": float(r1c["n_prims"].sum()) / dt_1,
              "ms_per_plan_p50": float(np.percentile(ro["device_ms"], 50)), "ms_per_plan_p95": float(np.percentile(ro["device_ms"], 95)),
              "sample": sample}
        if "reference_error" in pls:
            cb["reference_unavailable"] = pls["reference_error"]
        if "reference" in pls:  # the reference's own sources: time them on the same sample and check them too
            rr, dt_ref, util_ref = time_cpu(pls["reference"], so, go, threads, order)
            for f in ("pops", "n_nodes", "pop_hash", "closed_hash", "cost"):
                a, b2 = rr[f], res_all[f][:n_s]
                assert np.array_equal(a, b2) or f == "cost" and np.array_equal(a[np.isfinite(a)], b2[np.isfinite(b2)]), ("reference", f)
            cb.update({"value": float(rr["n_prims"].sum()) / dt_ref, "kind": "reference", "what": KIND_NOTE["reference"],
                       "thread_utilisation": util_ref, "port_value": port_v,
                       "ms_per_plan_p50": float(np.percentile(rr["device_ms"], 50)),
                       "ms_per_plan_p95": float(np.percentile(rr["device_ms"], 95))})
            cb["sample"] += " and against the reference's own sources"
        line["cpu_baseline"] = cb
    print(json.dumps(line))
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
