#!/usr/bin/env python
"""bench.py -- converged trajectories/sec of the batched MINCO/ALM optimizer (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W [--config 2|3|4|5]   # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K ...            # the reference algorithm on the host CPU cores (oracle)

A "step" is one pass of the hot path (B independent optimizeSE2Traj solves) over one batch of synthetic problems.  The default
workload is BASELINE.json configs[1] (the configuration the metric is quoted on): B = 1024 random SE(2) start/goal pairs per GPU
on the hill UnevenMap (weak scaling).  --config 3: 8192 problems on the desert map, STRONG scaling (8192 / N per GPU);
--config 4: volcano, max_kap 0.3, 64 samples per piece, B = 1024; --config 5: forest (run_forest.yaml), B = 4096.

The steps are PIPELINED over `--depth` lanes of one context (include/ualm.h: several batches in flight): step s+1 is launched
while the slowest trajectories of step s still run, and every step's results are complete inside the timed region.  `value` is
measured with the problems resident in HBM; `e2e` goes through the host-buffer C-ABI calls (ualm_submit_batch / ualm_wait_batch)
with pinned host inputs, H2D and D2H inside the timed region.  One JSON line on stdout (rank 0).

--dump-outputs DIR writes what the headline path returned in its last timed step (rank 0's shard): the coefficient vectors
c_xy / c_yaw and one array per result field, float64 .npy files, a fixed seeded sample of trajectories when they exceed 64 MB.
The inputs depend only on the arguments, so two builds can be compared output for output.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True          # the tree may be read-only: no __pycache__ next to the sources

METRIC = "converged trajectories/sec (batch MINCO)"
UNIT = "traj/s"
ROUND = "r02"


_T0 = time.perf_counter()


def note(msg):
    """progress on stderr (stdout carries the one JSON line)"""
    sys.stderr.write("[bench %7.1f s] %s\n" % (time.perf_counter() - _T0, msg))
    sys.stderr.flush()


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return json.load(open(p)).get("hbm_gbs", 6650.0), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def load_traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum per launch from THIS round's committed ncu --set full capture
    (profiles/traffic_r02.json names the command and the problem set it was taken on); absent -> null in the line."""
    p = os.path.join(ROOT, "profiles", "traffic_%s.json" % ROUND)
    if os.path.exists(p):
        return json.load(open(p))
    return {}


def usable_cores():
    """host threads this process may actually use: scheduler affinity, capped by the cgroup CPU quota"""
    n = len(os.sched_getaffinity(0))
    quota = None
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            quota = float(q) / float(per)
    except Exception:
        pass
    eff = n if quota is None else max(1, min(n, int(quota + 0.5)))
    return eff, {"os_cpu_count": os.cpu_count(), "sched_affinity": n, "cgroup_cpu_quota": quota}


def get_map(name):
    from uneven_planner_b200 import maps
    m = maps.get_terrain(name)
    if m is not None:
        return m, name
    # no .umap travelled: clearly labelled analytic stand-in (not one of the reference's terrains)
    return maps.synthetic_terrain("bumps", seed=0), "synthetic-bumps (maps_built/%s.umap missing)" % name


def make_problems(args, m, total, gen):
    from uneven_planner_b200 import problems
    if getattr(args, "front_end", "dubins") == "astar":
        return problems.generate_astar(m, total, seed=args.seed, **gen)
    return problems.generate(m, total, seed=args.seed, **gen)


def workload(args, world):
    """(terrain, params, generator kwargs, per-GPU batch, total batch, scaling, description) of the selected BASELINE config"""
    from uneven_planner_b200 import configs
    cfg = configs.BASELINE_CONFIGS[args.config]
    terrain = args.map or cfg["terrain"]
    total = (args.batch or cfg["batch"]) * (world if cfg["scaling"] == "weak" else 1)
    params = configs.params_for(terrain)
    desc = "configs[%d]: %d random SE(2) start/goal pairs%s on the %s UnevenMap, %s parameters%s" % (
        args.config - 1, total if cfg["scaling"] == "strong" else total // world, "" if cfg["scaling"] == "strong" else " per GPU", terrain,
        configs.YAML[terrain], "".join(", %s=%s" % kv for kv in configs.CONFIG_OVERRIDES.get(terrain, {}).items()))
    return terrain, params, configs.gen_kwargs(terrain), total, cfg["scaling"], desc


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index):
        self.index = index
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None

    def start(self):
        q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
            "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q, "--format=csv,noheader,nounits", "-lms", "100"],
                                      stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        rows = [l.strip().split(", ") for l in open(self.f.name) if l.strip()]
        os.unlink(self.f.name)
        sm, mx, reasons = [], [], set()
        for r in rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                    if v.strip().lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons),
                "samples": len(sm)}


def algorithmic_bytes(pb, res, K, e=8):
    """SURVEY 8d / BASELINE.md section 2: bytes the launch must move, from the work it actually did."""
    N = pb.N.astype(np.float64); M = pb.M.astype(np.float64)
    n = 1 + 2 * (N - 1) + (M - 1); S = N * (K + 1)
    evals = np.array([r.n_evals for r in res], dtype=np.float64)
    iters = np.array([r.n_lbfgs_iters for r in res], dtype=np.float64)
    sumb = np.array([r.sum_bound for r in res], dtype=np.float64)
    pen = evals * (S * 45 * e + (25 * N + 13 * M) * e)
    lb = (4 * n * sumb + 8 * n * iters) * e
    minco = evals * (n + 2 * (12 * N + 6 * M) + (N + M)) * e
    return float(pen.sum()), float(lb.sum()), float(minco.sum())


def time_reference_build(m, params, pb, threads, nprob=16):
    """oracle/_ref/libref.so = the reference's own alm_traj_opt.cpp compiled against oracle/shim (DESIGN.md section 8): timed on a few
    problems for the record.  It is bit-identical to the oracle port but several times slower (the shim evaluates every Eigen
    expression into heap temporaries), so the port stays the quoted CPU baseline."""
    path = os.path.join(ROOT, "oracle", "_ref", "libref.so")
    if not os.path.exists(path):
        return {"unavailable": "oracle/_ref/libref.so not built (needs the reference sources at build time)"}
    from concurrent.futures import ThreadPoolExecutor
    L = C.CDLL(path)
    dp = C.POINTER(C.c_double)
    L.ref_map_create.restype = C.c_void_p
    L.ref_alm_solve_h.restype = C.c_int
    L.ref_map_destroy.argtypes = [C.c_void_p]

    class RefParams(C.Structure):
        _fields_ = [(n, C.c_double) for n in ("rho_T", "rho_ter", "max_vel", "max_acc_lon", "max_acc_lat", "max_kap", "min_cxi", "max_sig")] + \
                   [("use_scaling", C.c_int)] + \
                   [(n, C.c_double) for n in ("rho", "beta", "gamma", "epsilon_con", "max_iter", "g_epsilon", "min_step", "inner_max_iter", "delta")] + \
                   [("mem_size", C.c_int), ("past", C.c_int), ("int_K", C.c_int), ("gravity", C.c_double)]
    rp = RefParams()
    for n, _ in RefParams._fields_:
        setattr(rp, n, getattr(params, n))
    g = m.geom
    cells = np.ascontiguousarray(m.cells, dtype=np.float64)
    vn = (C.c_int * 3)(*g.voxel_num); org = (C.c_double * 3)(*g.origin); mxb = (C.c_double * 3)(*g.max_boundary)
    nprob = min(nprob, pb.B)
    oxy, oyaw, _, _ = pb.offsets()
    # the reference prints from initScaling / the ALM loop: keep this process's stdout (one JSON line) clean
    sys.stdout.flush()
    saved = os.dup(1)
    devnull = os.open(os.devnull, os.O_WRONLY)
    os.dup2(devnull, 1)
    try:
        h = C.c_void_p(L.ref_map_create(cells.ctypes.data_as(dp), vn, org, mxb, C.c_double(g.xy_resolution), C.c_double(g.yaw_resolution),
                                        C.c_double(params.gravity)))

        def one(i):
            N, M = int(pb.N[i]), int(pb.M[i])
            S = N * (params.int_K + 1)
            ixy = np.ascontiguousarray(pb.inner_xy[oxy[i]:oxy[i + 1]]); iyaw = np.ascontiguousarray(pb.inner_yaw[oyaw[i]:oyaw[i + 1]])
            bufs = [np.zeros(k) for k in (12 * N, 6 * M, 2, S, 6 * S, S, 6 * S, 1, 7 * S, 1, 7)]
            bnd = np.ascontiguousarray(pb.bnd[i])
            return L.ref_alm_solve_h(C.byref(rp), h, N, M, bnd.ctypes.data_as(dp), C.c_double(float(pb.total_time[i])),
                                     (ixy if ixy.size else np.zeros(1)).ctypes.data_as(dp), (iyaw if iyaw.size else np.zeros(1)).ctypes.data_as(dp),
                                     *[b.ctypes.data_as(dp) for b in bufs])
        t0 = time.perf_counter()
        with ThreadPoolExecutor(min(threads, nprob)) as ex:
            rets = list(ex.map(one, range(nprob)))
        dt = time.perf_counter() - t0
        L.ref_map_destroy(h)
    finally:
        sys.stdout.flush()
        os.dup2(saved, 1)
        os.close(saved); os.close(devnull)
    return {"kind": "reference sources (alm_traj_opt.cpp, unmodified) against oracle/shim", "problems": nprob, "threads": min(threads, nprob),
            "converged_per_s": sum(1 for r in rets if r == 0) / dt, "seconds_per_trajectory_per_thread": dt / max(1, -(-nprob // min(threads, nprob))),
            "note": "bit-identical to the oracle port (tests/test_ref_pin.py); slower only because the Eigen stand-in is eager"}


DUMP_LIMIT = 64 << 20


def dump_outputs(path, res, cxy, cyaw, pb):
    """DIR/<name>.npy of one solved batch: c_xy, c_yaw and every ualm_result_t field, all float64.  Over DUMP_LIMIT bytes, a fixed seeded
    sample of whole trajectories is written instead, with their problem indices in sample_index.npy."""
    from uneven_planner_b200 import api
    fields = [f for f, _ in api.Result._fields_ if f != "reserved"]
    per = 8 * (12 * pb.N.astype(np.int64) + 6 * pb.M.astype(np.int64) + len(fields) + 1)
    idx = np.arange(pb.B)
    if per.sum() > DUMP_LIMIT:
        order = np.random.default_rng(0).permutation(pb.B)
        idx = np.sort(order[np.cumsum(per[order]) <= DUMP_LIMIT])
    _, _, ocx, ocy = pb.offsets()
    out = {"c_xy": np.concatenate([cxy[ocx[i]:ocx[i + 1]] for i in idx]) if len(idx) else np.zeros(0),
           "c_yaw": np.concatenate([cyaw[ocy[i]:ocy[i + 1]] for i in idx]) if len(idx) else np.zeros(0)}
    for f in fields:
        out[f] = np.array([getattr(res[i], f) for i in idx], dtype=np.float64)
    if len(idx) < pb.B:
        out["sample_index"] = idx.astype(np.float64)
    os.makedirs(path, exist_ok=True)
    for k, v in out.items():
        np.save(os.path.join(path, k + ".npy"), v)
    note("wrote %d arrays of %d trajectories to %s" % (len(out), len(idx), path))


def cpu_parallel_run(po, params, m, pb, threads):
    """the oracle on `threads` host threads over pb: (converged/s, seconds, converged count, mean in-thread seconds per trajectory)"""
    t0 = time.perf_counter()
    out = po.solve_batch(po.params_from(params), po.OracleMap(m), pb, threads=threads)
    dt = time.perf_counter() - t0
    conv = sum(1 for r in out if r[0].ret_code == 0)
    return conv / dt, dt, conv, float(np.mean([r[0].t_total for r in out]))


def run_reference(args):
    """--impl reference: the reference algorithm (CPU oracle port of alm_traj_opt.cpp, oracle/oracle.cpp) on all usable host cores, on the
    SAME workload as the CUDA arm (same terrain, parameters, seed; the whole batch per step unless --ref-sample bounds it).  Rank 0 only."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import pyoracle as po
    from uneven_planner_b200 import problems
    po.build()
    world = max(args.gpus, 1)
    terrain, params, gen, total, scaling, desc = workload(args, world)
    m, mname = get_map(terrain)
    threads, core_info = usable_cores()
    pb_all = make_problems(args, m, total, gen)
    sample = total if args.ref_sample <= 0 else min(args.ref_sample, total)
    pb = pb_all if sample == total else pb_all.select(np.arange(sample))
    for _ in range(min(args.warmup, 1)):
        po.solve_batch(po.params_from(params), po.OracleMap(m), pb.select(np.arange(min(threads, sample))), threads=threads)
    t0 = time.perf_counter()
    conv = 0
    for _ in range(args.steps):
        v, _, c, _ = cpu_parallel_run(po, params, m, pb, threads)
        conv += c
    dt = time.perf_counter() - t0
    val = conv / dt
    ref_build = time_reference_build(m, params, pb, threads)
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": scaling, "vs_baseline": None, "dtype": "f64",
            "data": "synthetic",
            "config": {"workload": desc.replace(terrain + " UnevenMap", mname + " UnevenMap") + ("" if args.front_end == "dubins" else "; initial paths from KinoAstar"), "global_batch": total, "batch_per_step": sample,
                       "same_config": sample == total,
                       "note": ("the whole batch per step" if sample == total else "a bounded sample of the batch per step: throughput is per trajectory, so the ratio stands") +
                               ", all usable host threads; inputs generated by libualm's HOST tools (Dubins + PlanManager resampler, no GPU code), the solve is oracle/liboracle.so"},
            "cpu_baseline": {"value": val, "unit": UNIT, "cores": threads, "cores_detail": core_info, "kind": "port",
                             "sample": "%d of the %d problems of the workload per step, %d host threads (one optimizer per thread)" % (sample, total, threads)},
            "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0, "reference_build": ref_build}
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=8, help="timed steps of every timed region (the throughput path's 8 lanes want 24 or more)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours")
    ap.add_argument("--config", type=int, default=2, choices=[2, 3, 4, 5], help="BASELINE.json config number (1-based)")
    ap.add_argument("--batch", type=int, default=0, help="override: problems per GPU per step (weak configs) / in total (config 3)")
    ap.add_argument("--map", default="", help="override the config's terrain")
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--front-end", default="dubins", choices=["dubins", "astar"], dest="front_end",
                    help="initial paths of the synthetic problems: one Dubins curve per pair (default, the workload every committed number uses) or the reference's own "
                         "front-end, KinoAstar::plan restated in libualm (ualm_front_end_batch)")
    ap.add_argument("--depth", type=int, default=0, help="batches in flight (lanes); 0 = 3 for the parity path, 8 for the throughput path; 1 = every step waits for its slowest trajectory")
    ap.add_argument("--precision", type=int, default=64, choices=[64, 65, 32], help="path of the HEADLINE numbers: 64 = parity path (default), 65 / 32 = throughput path")
    ap.add_argument("--no-fast", action="store_true", help="skip the separately labelled throughput-path measurement")
    ap.add_argument("--ref-sample", type=int, default=0, dest="ref_sample", help="reference arm / cpu_baseline: problems per step (0 = the whole batch, bounded at 1024 for cpu_baseline)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the un-pipelined latency datapoint and the penalty-kernel timing")
    ap.add_argument("--dump-outputs", default="", dest="dump_outputs", metavar="DIR",
                    help="write the results of the last timed step of the headline path to DIR/<name>.npy")
    args = ap.parse_args()
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as dist
    from uneven_planner_b200 import api, problems, distributed as D

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the product path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    dev = torch.device("cuda", local_rank)

    terrain, params, gen, Btot, scaling, desc = workload(args, world)
    m, mname = get_map(terrain)
    K = params.int_K
    pb_all = make_problems(args, m, Btot, gen)          # identical on every rank (counter-based RNG)
    shards = D.shard_indices(pb_all.nsamples(K), world)
    pb = pb_all.select(shards[rank])
    stride = D.record_stride(pb_all.N.max(), pb_all.M.max())

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def pinned(a):
        t = torch.from_numpy(np.ascontiguousarray(a)).pin_memory()
        return t, t.numpy()
    keep = [pinned(a) for a in (pb.N.astype(np.int32), pb.M.astype(np.int32), pb.bnd, pb.total_time, pb.inner_xy, pb.inner_yaw)]
    host_in = [k[1] for k in keep]
    h2d = int(sum(a.nbytes for a in host_in))

    def measure(precision, depth, steps, warmup, with_clocks, dump=False):
        """`value` (problems resident in HBM, steps pipelined over `depth` lanes) and `e2e` (host buffers through ualm_submit_batch /
        ualm_wait_batch) of one context of the given precision.  Returns a dict; the context stays open in r["opt"]."""
        opt = api.BatchALMTrajOpt(device=local_rank, precision=precision).init(params).set_environment(m)
        records = [torch.zeros((pb.B, stride), dtype=torch.float64, device=dev) for _ in range(depth)]
        full = [None]

        def collect(lane):
            """complete the step that ran on `lane` (host wait on the lane; the throughput engine advances every batch in flight
            meanwhile), pack its result records on the device, then the NCCL all-gather"""
            opt.select_lane(lane)
            opt.sync()
            opt.pack_records(records[lane].data_ptr(), stride)
            full[0] = D.all_gather_records(records[lane], shards, rank, world) if world > 1 else records[lane]

        def run_steps(nsteps):
            """nsteps passes over the resident batch, `depth` of them in flight; every step is complete when this returns"""
            for s in range(nsteps):
                lane = s % depth
                if s >= depth:
                    collect(lane)
                opt.select_lane(lane)
                if s == 0:
                    opt.mark_begin()
                opt.solve_resident()
            for s in range(max(0, nsteps - depth), nsteps):
                collect(s % depth)
            opt.select_lane(0)

        for lane in range(depth):
            opt.select_lane(lane)
            opt.upload(pb)
        note("precision %d: uploaded, warm-up" % precision)
        run_steps(max(warmup, 1))
        barrier()
        note("precision %d: timed region (%d steps, depth %d)" % (precision, steps, depth))
        sampler = ClockSampler(local_rank)
        if rank == 0 and with_clocks:
            sampler.start()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record()
        run_steps(steps)
        e1.record()
        barrier()
        clocks = sampler.stop() if (rank == 0 and with_clocks) else None
        ms = e0.elapsed_time(e1)
        lanes_ms = opt.mark_end()                  # CUDA events on the library's own streams: first launch -> last solve done
        tms = torch.tensor([ms], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tms, op=dist.ReduceOp.MAX)
        ms = float(tms.item())
        last = None
        if dump:
            opt.select_lane((steps - 1) % depth)
            last = opt.download()
        opt.select_lane(0)
        _, launches = opt.last_solve_ms()
        res, cxy, cyaw = opt.download()
        conv_local = sum(1 for r in res if r.ret_code == 0)
        full_h = full[0].cpu().numpy()
        conv_total = int((full_h[:, 0] == 0).sum()) if world > 1 else conv_local

        # e2e: host buffers through the C-ABI calls, H2D + D2H inside the timed region, `depth` batches in flight
        outs = []
        for _ in range(depth):
            _t1, o_cxy = pinned(np.zeros(int(12 * pb.N.astype(np.int64).sum())))
            _t2, o_cyaw = pinned(np.zeros(int(6 * pb.M.astype(np.int64).sum())))
            outs.append(((api.Result * pb.B)(), o_cxy, o_cyaw, _t1, _t2))

        def run_e2e(nsteps):
            tickets, conv = [], 0
            for s in range(nsteps):
                if s >= depth:
                    r, _, _ = opt.wait(tickets[s - depth], out=outs[s % depth][:3])
                    conv += sum(1 for q in r if q.ret_code == 0)
                tickets.append(opt.submit(pb, depth=depth, host=host_in))
            for s in range(max(0, nsteps - depth), nsteps):
                r, _, _ = opt.wait(tickets[s], out=outs[s % depth][:3])
                conv += sum(1 for q in r if q.ret_code == 0)
            return conv
        e2e_steps = steps
        note("precision %d: value done (%.1f ms/step), e2e" % (precision, ms / steps))
        run_e2e(depth)
        barrier()
        t0 = time.perf_counter()
        conv_e2e = run_e2e(e2e_steps)
        barrier()
        e2e_s = time.perf_counter() - t0
        te = torch.tensor([e2e_s, float(conv_e2e)], dtype=torch.float64, device=dev)
        if world > 1:
            tmax = te.clone(); dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
            dist.all_reduce(te, op=dist.ReduceOp.SUM)
            e2e_s, conv_e2e = float(tmax[0].item()), float(te[1].item())
        d2h = int(C.sizeof(api.Result) * pb.B + outs[0][1].nbytes + outs[0][2].nbytes)
        return dict(opt=opt, ms=ms, lanes_ms=lanes_ms, value=conv_total * steps / (ms * 1e-3), conv_total=conv_total, conv_local=conv_local,
                    res=res, last=last, launches=launches, clocks=clocks, depth=depth, steps=steps,
                    e2e={"value": conv_e2e / e2e_s, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "steps": e2e_steps,
                         "api": "ualm_submit_batch / ualm_wait_batch, pinned host buffers, %d batches in flight" % depth})

    def quality_of(opt, res):
        """independent check of a solved, collected batch (outside the timed region): the reference's post-solve scan
        (getMaxVxAxAyCurAttSig + getNonHolError, 0.01 s sampling) on the GPU, rank-local"""
        feas = opt.feasibility(0.01)
        okc = np.array([r.ret_code == 0 for r in res]) & (feas[:, 7] >= 0)
        tol = 1.05
        within = (np.abs(feas[:, 0]) <= params.max_vel * tol) & (np.abs(feas[:, 1]) <= params.max_acc_lon * tol) & \
                 (np.abs(feas[:, 2]) <= params.max_acc_lat * tol) & (np.abs(feas[:, 3]) <= params.max_kap * tol) & \
                 (-feas[:, 4] >= params.min_cxi / tol) & (feas[:, 5] <= params.max_sig * tol)
        return {"converged": int(okc.sum()), "converged_and_within_limits": int((okc & within).sum()),
                "limits": "max |vx|, |ax|, |ay|, |curvature|, sigma <= 1.05 x limit and min cos(xi) >= limit / 1.05 over 0.01 s samples "
                          "(ualm_feasibility_batch; rank 0's shard)",
                "median_nonholonomic_error_per_sample": float(np.median(feas[okc, 6] / np.maximum(feas[okc, 7], 1.0))) if okc.any() else None}

    # ---------------- the headline: the parity path (precision 64, bit-identical to the oracle) ----------------
    head_prec = args.precision
    depth = max(1, min(args.depth if args.depth > 0 else (3 if head_prec == 64 else 8), 8))
    r0 = measure(head_prec, depth, args.steps, args.warmup, True, dump=bool(args.dump_outputs))
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, *r0["last"], pb)
    opt, res, ms, lanes_ms, value, conv_total, conv_local, launches, clocks = (r0[k] for k in ("opt", "res", "ms", "lanes_ms", "value", "conv_total", "conv_local", "launches", "clocks"))
    opt.select_lane(0)
    quality = quality_of(opt, res)

    # ---------------- roofline of the dominant kernel(s) over the timed region ----------------
    peak, peak_src = load_peaks()
    traffic = load_traffic()

    def roofline_of(r, precision):
        e = 4 if precision == 32 else 8
        pen_b, lb_b, mc_b = algorithmic_bytes(pb, r["res"], K, e)
        mc_b = mc_b * 8 / e                                                  # the MINCO vectors stay double on every path
        alg = pen_b + lb_b + mc_b
        step_ms = r["lanes_ms"] / r["steps"]                                 # the kernels of consecutive steps overlap: average per step
        achieved = alg / (step_ms * 1e-3) / 1e9
        if precision == 64:
            kern = "ualm::solve_kernel (whole ALM/L-BFGS solve of the batch: a warp group per trajectory, one launch per size class on concurrent streams, %d batches in flight)" % r["depth"]
            note = "latency-bound: bit-reproducible fp64 dependent chains, a warp group per trajectory (DESIGN.md section 4)"
            key = "solve_kernel_bytes_per_launch_config%d" % args.config
        else:
            kern = "ualm_tp::ka_kernel + kb_kernel rounds (one evaluation of every active trajectory per round, %d batches in flight, every batch its own stream)" % r["depth"]
            note = "ka_kernel: warp per trajectory, latency-bound serial sweeps / two-loop; kb_kernel: thread per sample (DESIGN.md section 4)"
            key = "tp_round_bytes_per_step_config%d" % args.config
        return {"kernel": kern, "bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": traffic.get(key), "traffic_source": traffic.get("source"), "peak_source": peak_src, "kernel_ms": step_ms,
                "algorithmic_bytes": {"penalty": pen_b, "lbfgs": lb_b, "minco_io": mc_b},
                "note": note + "; kernel_ms = CUDA-event time of the timed region on the library's own streams / steps"}

    def penalty_roofline(o, precision):
        if precision == 64:
            pms, pbytes = o.time_penalty_kernel(5)
            return {"kernel": "ualm::penalty_only_kernel (calConstrainCostGrad samples + accumulation, 1 evaluation per trajectory)",
                    "bound": "hbm", "achieved": pbytes / (pms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s", "frac": pbytes / (pms * 1e-3) / 1e9 / peak,
                    "traffic": traffic.get("penalty_only_kernel_bytes_per_launch_config%d" % args.config), "kernel_ms": pms}
        out = {}
        for tma in (1, 0):
            os.environ["UALM_TP_TMA"] = "1" if tma else "0"
            pms, pbytes = o.time_penalty_kernel(10)
            out["tma_tiles" if tma else "direct_gather (default)"] = {"kernel_ms": pms, "achieved": pbytes / (pms * 1e-3) / 1e9, "frac": pbytes / (pms * 1e-3) / 1e9 / peak}
        os.environ.pop("UALM_TP_TMA", None)
        best = max(out.values(), key=lambda v: v["achieved"])
        return {"kernel": "ualm_tp::kb_kernel<%s> (calConstrainCostGrad: thread per sample, CTA per trajectory, 1 evaluation per trajectory, the whole batch in one launch)" % ("float" if precision == 32 else "double"),
                "bound": "hbm", "achieved": best["achieved"], "peak": peak, "unit": "GB/s", "frac": best["frac"], "kernel_ms": best["kernel_ms"],
                "algorithmic_bytes": pbytes, "variants": out, "traffic": traffic.get("kb_kernel_bytes_per_launch_config%d" % args.config)}

    roof = roofline_of(r0, head_prec)
    step_ms = roof["kernel_ms"]
    extras = None
    roof_pen = None
    if not args.no_extras:
        # one un-pipelined solve (latency of a batch = its slowest trajectory) and the penalty phase alone, outside the timed region
        opt.select_lane(0)
        opt.solve_resident(); opt.sync()
        single_ms, _ = opt.last_solve_ms()
        extras = {"single_batch_ms": single_ms, "single_batch_converged_per_s": conv_local / single_ms * 1e3,
                  "note": "one batch alone on the device (depth 1): bounded by its slowest trajectory"}
        roof_pen = penalty_roofline(opt, head_prec)
    opt.close()

    # ---------------- the throughput path (precision 32), separately labelled; the headline above stays on the parity path ----------------
    fast = None
    if head_prec == 64 and not args.no_fast:
        fdepth = 8
        # the timed region starts and ends with an empty pipeline (synchronize on both sides), so fewer steps than about three times the
        # eight lanes mostly measure filling and draining them
        rf = measure(32, fdepth, args.steps, max(args.warmup, fdepth), False)
        fo = rf["opt"]
        fo.select_lane(0)
        note("fast path measured; post-solve scan")
        fq = quality_of(fo, rf["res"])
        fev = np.array([r.n_evals for r in rf["res"]])
        fo.select_lane(0); fo.upload(pb)
        fpen = None if args.no_extras else penalty_roofline(fo, 32)
        fast = {"precision": 32, "what": "throughput path (ualm_create(precision = 32)): lockstep evaluation rounds with continuous batching, penalty samples in float, "
                                         "solver state in double; NOT bit-comparable with the oracle (tests/test_gpu_tp.py bounds one evaluation; profiles/config5_sweep_%s.json "
                                         "holds the end-to-end distribution)" % ROUND,
                "value": rf["value"], "solved_per_s": Btot * rf["steps"] / (rf["ms"] * 1e-3), "unit": UNIT, "ms_per_step": rf["ms"] / rf["steps"], "steps": rf["steps"], "batches_in_flight": fdepth,
                "e2e": rf["e2e"], "converged_per_step": rf["conv_total"], "speedup_vs_parity_path": rf["value"] / value if value > 0 else None,
                "quality": fq, "evals_per_step": int(fev.sum()), "roofline": roofline_of(rf, 32), "roofline_penalty": fpen,
                "note": None if rf["steps"] >= 3 * fdepth else
                        "%d timed steps over %d lanes: the figure is dominated by filling and draining the pipeline; --steps %d or more measures "
                        "the steady state" % (rf["steps"], fdepth, 3 * fdepth)}
        fo.close()

    # ---------------- CPU baseline on this box's host cores (rank 0, bounded sample) ----------------
    note("GPU arms done; cpu baseline")
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        sys.path.insert(0, os.path.join(ROOT, "oracle"))
        import pyoracle as po
        po.build()
        threads, core_info = usable_cores()
        sample = min(args.ref_sample if args.ref_sample > 0 else 1024, pb_all.B)
        sub = pb_all.select(np.arange(sample))
        cpu_v, dt, cpu_conv, one = cpu_parallel_run(po, params, m, sub, threads)
        # the reference's own operating mode: one optimizer on one otherwise idle core (SURVEY 8d: "1 thread, per-trajectory ms")
        n1 = min(8, sample)
        t1 = time.perf_counter()
        o1 = po.solve_batch(po.params_from(params), po.OracleMap(m), pb_all.select(np.arange(n1)), threads=1)
        one_idle = (time.perf_counter() - t1) / n1
        conv1 = sum(1 for r in o1 if r[0].ret_code == 0) / max(n1, 1)
        solved_per_s = sample / dt
        cpu = {"value": cpu_v, "unit": UNIT, "cores": threads, "cores_detail": core_info, "kind": "port",
               "single_thread_ms_per_trajectory": one_idle * 1e3,
               "parallel_efficiency": solved_per_s / (threads / one_idle) if one_idle > 0 else None,
               "sample": "first %d problems of the workload, %d host threads (one optimizer instance per thread), %.1f s; mean %.1f ms/trajectory inside a "
                         "thread under that load, %.1f ms/trajectory for the first %d problems on one thread of the idle host (converged fraction %.2f)"
                         % (sample, threads, dt, one * 1e3, one_idle * 1e3, n1, conv1)}

    if rank == 0:
        ev = np.array([r.n_evals for r in res])
        slow = int(np.argmax(ev))
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": scaling, "vs_baseline": None,
                "dtype": "f64" if head_prec != 32 else "f32 penalty samples / f64 solver state",
                "data": "synthetic",
                "config": {"workload": desc.replace(terrain + " UnevenMap", mname + " UnevenMap") + ("" if args.front_end == "dubins" else "; initial paths from KinoAstar"), "precision": head_prec,
                           "global_batch": Btot, "parallelism": "dp%d (independent shards, final NCCL all-gather of result records)" % world,
                           "converged_per_step": conv_total, "solved_per_step": Btot, "batches_in_flight": depth,
                           "pipelining": "steps are launched on %d lanes round robin; a lane is re-used only after its previous step is complete; all %d steps "
                                         "are complete (results packed%s) inside the timed region" % (depth, args.steps, ", all-gathered" if world > 1 else ""),
                           "l2": "no flush needed: per-step working set (L-BFGS history + sample scratch, %.0f MB per lane) exceeds the 126 MB L2; the 41 MB map is "
                                 "reused within a step" % ((8.0 * 2 * params.mem_size * float(pb.nvar().sum())) / 1e6)},
                "e2e": r0["e2e"], "solved_per_s": Btot * args.steps / (ms * 1e-3),
                "gpu_launches": int((launches + 1) * args.steps),
                "clocks": clocks, "roofline": roof, "roofline_penalty": roof_pen, "cpu_baseline": cpu, "latency": extras, "quality": quality,
                "fast_path": fast,
                "work": {"evals_per_step": int(ev.sum()), "lbfgs_iters_per_step": int(sum(r.n_lbfgs_iters for r in res)), "rank0_batch": pb.B,
                         "evals_per_trajectory": {"mean": float(ev.mean()), "p50": float(np.percentile(ev, 50)), "p99": float(np.percentile(ev, 99)),
                                                  "second_max": int(np.sort(ev)[-2]) if len(ev) > 1 else int(ev.max()), "max": int(ev.max())},
                         "slowest_trajectory": {"n_evals": int(ev[slow]), "N": int(pb.N[slow]), "ret_code": int(res[slow].ret_code),
                                                "outer_iters": int(res[slow].outer_iters)},
                         "lanes_event_ms_per_step": step_ms}}
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
