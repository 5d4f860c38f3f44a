#!/usr/bin/env python
"""bench.py -- the hot path of BASELINE.json on N B200s of one node.

Workload (config.workload): a sweep of synthetic cavity pairs shaped like the BO1 dataset (BASELINE.json configs[4]
shape, per-pair settings of configs[1]: the shipped config.txt with its incompatibility term, Nd = all source points,
DT 20^3), `--pairs` pairs per GPU per step (weak scaling: pairs are sharded across ranks, no data-path collective).
One step = BuildDT + Initialize + Register of every pair of the rank's block.

  value     cube.point bound evals / s (1 eval = jly_goicp.cpp:369-381 once), whole job, inputs resident in HBM
  e2e       the same through the C-ABI call that takes HOST buffers (goicp_register_batch): host preprocessing,
            host->device copies and the result read-back inside the timed region
  roofline  dominant kernel = search_kernel (the device-resident search: OuterBnB + every InnerBnB call + ICP of the whole
            batch in one launch); achieved = evals x algorithmic bytes per eval (SURVEY 8(d)) / its CUDA-event time,
            against the measured HBM copy peak (MEASURED_PEAKS.json)
  cpu_baseline  the reference's own CPU implementation (oracle/_ref, compiled from its sources) on a bounded sample
            of the same pairs, one process per host core, longest pairs first
  per_pair  BASELINE metric #2 (wall time per registration pair) for configs 1-4 at their full sizes, GPU (DT build, Register)
            beside the single-core reference

`--impl reference` times the CPU arm alone on the same config/metric.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
METRIC, UNIT = "cube_point_bound_evals_per_sec", "evals/s"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--pairs", type=int, default=4096, help="cavity pairs per GPU per step")
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--exact", type=int, default=1, help="1: reference-identical sequential float sums; 0: warp-tree sums")
    ap.add_argument("--fpfh", type=int, default=0, help="1: add the c-FPFH term (cfpfh=1, regularizationFPFH=5e-6)")
    ap.add_argument("--cpu-pairs", type=int, default=0, help="pairs in the CPU-baseline sample (0: 16 per core)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-per-pair", action="store_true", help="skip the per-pair wall times of configs 1-4")
    ap.add_argument("--per-pair-cpu-deep", action="store_true", help="also time the reference on config 4 at 512^3 (several minutes of one core)")
    ap.add_argument("--workload", default="sweep", choices=["sweep", "deep"], help="sweep: the BO1-shaped batch (headline); deep: ONE deep registration (BASELINE config 4) "
                    "in relaxed-order wave mode, the InnerBnB calls of every wave sharded over the ranks (strong scaling)")
    ap.add_argument("--wave-nodes", type=int, default=256, help="deep workload: rotation nodes expanded per wave")
    ap.add_argument("--seed", type=int, default=4096)
    ap.add_argument("--groups", type=int, default=-1, help="wave scheduler only: worker streams per GPU (-1: library default)")
    ap.add_argument("--slots", type=int, default=-1, help="wave scheduler only: pairs advanced in lock-step per stream (-1: library default)")
    ap.add_argument("--spec", type=int, default=-1, help="wave scheduler only: speculation width in rotation nodes (-1: library default)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the registrations of rank 0's last timed step as DIR/<name>.npy (see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes what the GPU arm computed; it does not apply to --impl reference")
    return args


DUMP_ROWS = 100000   # 172 B per registration: two dumped legs stay under 64 MB


def dump_outputs(out_dir, results, prefix=""):
    """The arrays a caller receives from one timed step, one row per registration: R (n,3,3), t (n,3), opt_error (n,),
    opt_comp (n,), status (n,), the search counters 0-5 of goicp_result (n,6) and index (n,), the row's position in the step.  Counters 6-7
    (launches, speculative re-runs) describe the schedule, not the result, and are left out.  A step of more than DUMP_ROWS
    registrations is written as a fixed, seeded sample of them.  The inputs are seeded too, so two builds run with the same
    arguments can be compared file for file."""
    idx = np.arange(len(results))
    if len(idx) > DUMP_ROWS:
        idx = np.sort(np.random.default_rng(0).choice(len(idx), DUMP_ROWS, replace=False))
    rows = [results[i] for i in idx]
    os.makedirs(out_dir, exist_ok=True)
    arrays = {"R": np.array([r["R"] for r in rows], np.float64).reshape(-1, 3, 3),
              "t": np.array([r["t"] for r in rows], np.float64).reshape(-1, 3),
              "opt_error": np.array([r["optError"] for r in rows], np.float32),
              "opt_comp": np.array([r["optComp"] for r in rows], np.float64),
              "status": np.array([r["status"] for r in rows], np.float64),
              "counters": np.array([list(r["counters"])[:6] for r in rows], np.float64).reshape(-1, 6),
              "index": idx.astype(np.float64)}
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, prefix + name + ".npy"), a)


def config_dict(args):
    return {"workload": "BO1-shaped synthetic cavity pairs (configs[4] shape; per-pair settings of configs[1]: shipped config.txt, "
                        "Nd=all, DT 20^3%s)" % (", c-FPFH term" if args.fpfh else ""),
            "pairs_per_gpu": args.pairs, "sharding": "pairs across ranks, no collective on the data path",
            "sums": "exact (reference order)" if args.exact else "warp-tree",
            "l2": "flushed between timed steps (256 MiB write)"}


# ---- CPU arm: the reference compiled from its own sources, one process per core -------------------------------------------------
def _cpu_worker(job):
    kind, pair, fpfh = job
    from oracle import pyoracle as po
    kw = dict(cfpfh=1, regularizationFPFH=0.000005) if fpfh else {}
    o = po.Oracle(kind, pair["model_xyz"], pair["data_xyz"], po.shipped_config(**kw), model_c=pair["model_c"], data_c=pair["data_c"],
                  model_fpfh=pair["model_fpfh"], data_fpfh=pair["data_fpfh"])
    t0 = time.perf_counter()
    r = o.register(pair["nd"])
    dt = time.perf_counter() - t0
    o.close()
    return r["counters"][2] * pair["nd"], r["optError"], dt


def cpu_arm(pairs, fpfh, cores, order=None):
    """The reference over `pairs` on `cores` worker processes fed from one queue, pairs in `order` (longest first when their cost
    is known: the makespan is then the work, not one deep pair).  Returns a dict."""
    import multiprocessing as mp
    from oracle import pyoracle as po
    kind = "ref" if po.available("ref") else "port"
    po._lib(kind)
    idx = list(range(len(pairs))) if order is None else list(order)
    jobs = [(kind, pairs[i], fpfh) for i in idx]
    ctx = mp.get_context("fork")
    with ctx.Pool(cores) as pool:
        pool.map(_cpu_worker, jobs[-cores:])   # touch pages / load libs in every worker (the cheapest pairs)
        t0 = time.perf_counter()
        out = list(pool.imap(_cpu_worker, jobs, chunksize=1))
        dt = time.perf_counter() - t0
    evals = float(sum(o[0] for o in out)); busy = float(sum(o[2] for o in out))
    errs = [None] * len(pairs); secs = [0.0] * len(pairs)
    for i, o in zip(idx, out):
        errs[i], secs[i] = o[1], o[2]
    return {"value": evals / dt, "seconds": dt, "kind": "reference" if kind == "ref" else "port", "opt_errors": errs, "pair_seconds": secs,
            "per_core": evals / busy, "busy_fraction": busy / (dt * cores), "evals": evals}


# ---- per-pair wall times of BASELINE configs 1-4 (metric #2) --------------------------------------------------------------------
def _pp_cases(g, synth):
    def golden(name):
        return np.load(os.path.join(ROOT, "tests", "golden", name + ".npz"))
    cases = []
    z = golden("bunny")
    cases.append(dict(name="config1 bunny (Nm 35947, Nd 1000, DT 300^3, MSE 1e-3)", model=z["model_xyz"], data=z["data_xyz"], nd=int(z["nd"]), cfg=("upstream", dict(distTransSize=300)), exp=float(z["exp300_optError"]), clouds={}))
    z = golden("pair1")
    cl = dict(model_c=z["model_c"], data_c=z["data_c"], model_fpfh=z["model_fpfh"], data_fpfh=z["data_fpfh"])
    cases.append(dict(name="config2 cavity pair 1 (2x86_3 -> 1eq2_6, Nd 238, shipped config.txt)", model=z["model_xyz"], data=z["data_xyz"], nd=int(z["nd"]), cfg=("shipped", {}), exp=float(z["exp_optError"]), clouds=cl))
    cases.append(dict(name="config2 cavity pair 1 + c-FPFH term", model=z["model_xyz"], data=z["data_xyz"], nd=int(z["nd"]), cfg=("shipped", dict(cfpfh=1, regularizationFPFH=0.000005)), exp=float(z["expf_optError"]), clouds=cl))
    z = golden("pair2")
    cl = dict(model_c=z["model_c"], data_c=z["data_c"], model_fpfh=z["model_fpfh"], data_fpfh=z["data_fpfh"])
    cases.append(dict(name="config2 cavity pair 2 (2ktd_1 -> 4imo_2, Nd 247: the deep cavity case)", model=z["model_xyz"], data=z["data_xyz"], nd=int(z["nd"]), cfg=("shipped", {}), exp=float(z["exp_optError"]), clouds=cl))
    z = golden("rand")
    cases.append(dict(name="config3 rand clouds (100 x 100, trimFraction 0.1, DT 300^3)", model=z["model_xyz"], data=z["data_xyz"], nd=int(z["nd"]), cfg=("upstream", dict(distTransSize=300, trimFraction=0.1)), exp=float(z["exp300_optError"]), clouds={}))
    p = synth.deep_pair(1236)
    cases.append(dict(name="config4 synthetic deep (Nm 100000, Nd 10000, DT 512^3, MSE 1e-4; seed 1236: the first ICP does not reach the optimum)", model=p["model_xyz"], data=p["data_xyz"], nd=10000,
                      cfg=("upstream", dict(distTransSize=512, MSEThresh=1e-4)), exp=None, clouds={}, deep=True))
    return cases


def _pp_cpu_worker(job):
    """single-core reference: (DT seconds, Register seconds, optError)"""
    kind, case = job
    from oracle import pyoracle as po
    params = (po.shipped_config if case["cfg"][0] == "shipped" else po.upstream_config)(**case["cfg"][1])
    o = po.Oracle(kind, case["model"], case["data"], params, **case["clouds"])
    t0 = time.perf_counter(); o.build_dt(); tdt = time.perf_counter() - t0
    t0 = time.perf_counter(); r = o.register(case["nd"]); treg = time.perf_counter() - t0
    o.close()
    return tdt, treg, r["optError"]


def per_pair_gpu(g, cases):
    out = []
    for c in cases:
        params = (g.shipped_config if c["cfg"][0] == "shipped" else g.upstream_config)(**c["cfg"][1])
        reg = g.GoICP(c["model"], c["data"], params, **c["clouds"])
        tdt, treg = [], []
        r = None
        for _ in range(3):
            t0 = time.perf_counter(); reg.BuildDT(); tdt.append(time.perf_counter() - t0)
            reg.set_nd(c["nd"])
            t0 = time.perf_counter(); r = reg.Register(); treg.append(time.perf_counter() - t0)
        out.append({"config": c["name"], "gpu_ms_dt": 1e3 * sorted(tdt)[1], "gpu_ms_register": 1e3 * sorted(treg)[1], "gpu_opt_error": r["optError"],
                    "sub_cubes": int(r["counters"][2]), "rotation_pops": int(r["counters"][3]), "evals": float(r["counters"][2]) * c["nd"]})
        del reg
    return out


class ClockSampler(threading.Thread):
    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.stop_flag, self.rows = index, False, []

    def run(self):
        q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q, "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([c.strip() for c in out.split(",")])
            except Exception:
                pass
            time.sleep(0.2)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unsampled"]}
        sm = sorted(int(r[0]) for r in self.rows if r[0].isdigit())
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for k, n in enumerate(names) if any(len(r) > 2 + k and r[2 + k].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": int(self.rows[0][1]) if self.rows[0][1].isdigit() else None, "reasons": reasons, "samples": len(self.rows)}


def reference_arm(args, synth, cores):
    """`--impl reference`: the reference CPU implementation alone, all host cores, same metric / config; each step a bounded sample of
    the workload sized so that the whole run ends within a few minutes (the first warm-up step measures every pair's cost, the
    following steps feed the workers longest pair first)."""
    budget_s = 150.0 / max(1, args.steps + args.warmup)              # wall seconds per step
    n = args.cpu_pairs or int(max(4 * cores, min(16 * cores, budget_s * cores * 1.6)))   # ~0.6 s of one core per pair on average
    pairs = synth.bo1_pairs(n, seed=args.seed)
    order, vals, t_all, last = None, [], 0.0, None
    for k in range(max(1, args.warmup)):
        last = cpu_arm(pairs, args.fpfh, cores, order)
        order = list(np.argsort(last["pair_seconds"])[::-1])
    for _ in range(args.steps):
        last = cpu_arm(pairs, args.fpfh, cores, order)
        vals.append(last["value"]); t_all += last["seconds"]
    val = float(np.mean(vals))
    sample = f"{n} pairs of the workload per step (seed {args.seed}), {cores} worker processes fed longest pair first from one queue; all cores busy {100 * last['busy_fraction']:.0f} % of the step"
    print(json.dumps({"impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
                      "ms_per_step": 1e3 * t_all / max(1, args.steps), "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32+f64",
                      "data": "synthetic", "config": config_dict(args),
                      "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": last["kind"], "sample": sample, "per_core": last["per_core"], "busy_fraction": last["busy_fraction"]},
                      "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))


def deep_arm(args, g, synth, rank, world, local):
    """`--workload deep`: SURVEY 8(e) second shard.  Every rank holds the same pair and its DT; the rotation frontier is advanced in
    waves of --wave-nodes nodes, each wave's InnerBnB calls are split over the ranks and the result records all-gathered, every rank
    applies them identically (same optimum, counters and trace on every rank: checked).  A step = one whole registration."""
    import torch
    import torch.distributed as dist
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)

    def golden(name):
        return np.load(os.path.join(ROOT, "tests", "golden", name + ".npz"))
    p = synth.deep_pair(1236)
    z2, zs = golden("pair2"), golden("deep_small")
    cases = [("config4 synthetic deep (Nm 100000, Nd 10000, DT 512^3, MSE 1e-4, seed 1236)", p["model_xyz"], p["data_xyz"], 10000, g.upstream_config(distTransSize=512, MSEThresh=1e-4), {}),
             ("config4 shape at 20000 x 2000, DT 128^3 (tests/golden/deep_small)", zs["model_xyz"], zs["data_xyz"], int(zs["nd"]), g.upstream_config(distTransSize=128, MSEThresh=1e-4), {}),
             ("cavity pair 2 (2ktd_1 -> 4imo_2, shipped config.txt)", z2["model_xyz"], z2["data_xyz"], int(z2["nd"]), g.shipped_config(),
              dict(model_c=z2["model_c"], data_c=z2["data_c"], model_fpfh=z2["model_fpfh"], data_fpfh=z2["data_fpfh"]))]
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    rows, last = [], []
    for name, m, d, nd, params, cl in cases:
        reg = g.GoICP(m, d, params, device=local, **cl)
        reg.BuildDT(); reg.set_nd(nd)
        exact, t_exact = None, None
        if rank == 0:    # the reference's visitation order on one GPU, for the comparison (before the sharding is switched on: no collective inside)
            reg.set_search_mode(0, -1)
            reg.Register()
            torch.cuda.synchronize(dev); t0 = time.perf_counter(); exact = reg.Register(); torch.cuda.synchronize(dev); t_exact = 1e3 * (time.perf_counter() - t0)
        if world > 1:
            dist.barrier()
            reg.eng.set_frontier_sharding(rank, world, dev)
        reg.set_search_mode(1, args.wave_nodes)
        for _ in range(args.warmup):
            reg.Register()
        ts, r = [], None
        for _ in range(args.steps):
            if world > 1:
                dist.barrier()
            torch.cuda.synchronize(dev)
            t0 = time.perf_counter(); r = reg.Register(); torch.cuda.synchronize(dev); ts.append(1e3 * (time.perf_counter() - t0))
        last.append(r)
        sig = torch.tensor([sum(ts), r["optError"]] + [float(v) for v in r["counters"][:6]], dtype=torch.float64, device=dev)
        same = True
        if world > 1:
            ref = sig.clone(); dist.broadcast(ref, 0); same = bool(torch.equal(ref[1:], sig[1:]))
            mx = sig.clone(); dist.all_reduce(mx, op=dist.ReduceOp.MAX); total_ms = mx[0].item()
            ok = torch.tensor([1.0 if same else 0.0], dtype=torch.float64, device=dev); dist.all_reduce(ok, op=dist.ReduceOp.MIN); same = bool(ok.item() > 0)
        else:
            total_ms = sum(ts)
        evals = float(r["counters"][2]) * nd
        rows.append({"case": name, "ms_per_registration": total_ms / args.steps, "evals_per_registration": evals, "value": evals * args.steps / (total_ms * 1e-3),
                     "opt_error": r["optError"], "rotation_pops": int(r["counters"][3]), "inner_calls": int(r["counters"][0]), "gpu_ms_bnb": r["gpu_ms_bnb"], "gpu_ms_icp": r["gpu_ms_icp"], "launches_per_registration": int(r["counters"][6]),
                     "same_result_on_every_rank": same,
                     "exact_order_1gpu": None if exact is None else {"ms": t_exact, "opt_error": exact["optError"], "rotation_pops": int(exact["counters"][3]), "inner_calls": int(exact["counters"][0])}})
        del reg
    sampler.stop_flag = True
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last)
    if rank == 0:
        h = rows[0]
        print(json.dumps({"metric": METRIC, "value": h["value"], "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": h["ms_per_registration"],
                          "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32+f64", "data": "synthetic",
                          "config": {"workload": "deep: " + h["case"] + "; relaxed-order waves of %d rotation nodes, calls sharded over %d rank(s), one all-gather of result records per wave; "
                                     "inputs resident (DT built before the timed region); ICP runs replicated on every rank" % (args.wave_nodes, world)},
                          "gpu_launches": int(rows[0]["launches_per_registration"]) * args.steps, "cases": rows, "clocks": sampler.summary()}))
    if world > 1:
        dist.destroy_process_group()


def main():
    args = parse()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    import __graft_entry__ as ge
    g = ge.load_package()
    import importlib
    synth = importlib.import_module("goicp_b200.synth")
    cores = os.cpu_count() or 1

    if args.impl == "reference":
        if rank == 0:
            reference_arm(args, synth, cores)
        return

    if args.workload == "deep":
        deep_arm(args, g, synth, rank, world, local)
        return

    import torch
    import torch.distributed as dist
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    stream = torch.cuda.current_stream(dev)
    eng = g.Engine(local, stream.cuda_stream)          # kernels run on torch's current stream: torch events see them
    eng.set_options(args.exact, args.spec, -1)
    eng.set_batch_options(args.groups, args.slots)
    kw = dict(cfpfh=1, regularizationFPFH=0.000005) if args.fpfh else {}
    params = g.shipped_config(**kw)
    pairs = synth.bo1_pairs(args.pairs, seed=args.seed + 7919 * rank)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def evals_of(res):
        return float(sum(r["counters"][2] * p["nd"] for r, p in zip(res, pairs)))

    # ---- resident leg: inputs uploaded before the timed region ----
    eng.batch_upload(params, pairs)
    for _ in range(args.warmup):
        flush.zero_()
        res = eng.batch_run()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    kern_ms, launches, total_evals = 0.0, 0, 0.0
    barrier()
    t0 = time.perf_counter()
    for k in range(args.steps):
        flush.zero_()
        ev[k][0].record(stream)
        res = eng.batch_run()
        ev[k][1].record(stream)
        tm = eng.timings()
        kern_ms += tm["ms"][2]; launches += sum(tm["launches"]); total_evals += evals_of(res)
        last_tm, last_stats = tm, eng.stats()
    barrier()
    wall = time.perf_counter() - t0
    dev_ms = sum(a.elapsed_time(b) for a, b in ev)
    # ---- e2e leg: host buffers in, results out, through the public C-ABI call ----
    descs = eng.make_descs(pairs)   # goicp_pair_desc[]: pointers to the host (numpy) buffers, built once like any C caller would
    for _ in range(min(args.warmup, 1)):
        eng.register_batch_descs(params, descs)
    barrier()
    e2e_ms, e2e_evals = 0.0, 0.0
    for k in range(args.steps):
        flush.zero_()
        torch.cuda.synchronize(dev)
        t1 = time.perf_counter()
        r2 = eng.register_batch_descs(params, descs)   # host buffers -> H2D -> DT build -> Register -> results in host memory
        torch.cuda.synchronize(dev)
        e2e_ms += 1e3 * (time.perf_counter() - t1); e2e_evals += float(sum(r.counters[2] * p["nd"] for r, p in zip(r2, pairs)))
    barrier()
    sampler.stop_flag = True
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, res)
        dump_outputs(args.dump_outputs, [g._result_dict(r) for r in r2], prefix="e2e_")
    h2d = sum(p[k].nbytes for p in pairs for k in ("model_xyz", "data_xyz", "model_c", "data_c")) + (sum(p["model_fpfh"].nbytes + p["data_fpfh"].nbytes for p in pairs) if args.fpfh else 0)
    d2h = len(pairs) * 208

    stats = torch.tensor([dev_ms, e2e_ms, total_evals, e2e_evals, kern_ms, float(launches)], dtype=torch.float64, device=dev)
    if world > 1:
        mx = stats.clone(); dist.all_reduce(mx, op=dist.ReduceOp.MAX)
        sm = stats.clone(); dist.all_reduce(sm, op=dist.ReduceOp.SUM)
        dev_ms, e2e_ms, kern_ms = mx[0].item(), mx[1].item(), mx[4].item()
        total_evals, e2e_evals, launches = sm[2].item(), sm[3].item(), int(sm[5].item())
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    value = total_evals / (dev_ms * 1e-3)
    peaks, peak_src = {"hbm_gbs": 6650.0}, "fallback"
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))); peak_src = "measured"
    except Exception:
        pass
    kern_evals_per_gpu = total_evals / world
    # SURVEY.md 8(d): 4 B per cube.point eval (one DT voxel) + with regularization>0 27/8 corner evals x (4 B index map + 2 B
    # property mask) = 20.25 B (+ 27/8 x 4 B of the per-cell c-FPFH table with the c-FPFH term)
    bytes_per_eval = 4.0 + (20.25 if params.regularization > 0 else 0.0) + (13.5 if args.fpfh else 0.0)
    achieved = kern_evals_per_gpu * bytes_per_eval / (kern_ms * 1e-3) / 1e9
    agg = total_evals / world * bytes_per_eval / (dev_ms * 1e-3) / 1e9
    roof = {"bound": "hbm", "kernel": "search_kernel", "achieved": achieved, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": achieved / peaks["hbm_gbs"],
            "traffic": None, "peak_source": peak_src, "achieved_aggregate": agg, "frac_aggregate": agg / peaks["hbm_gbs"],
            "algorithmic_bytes_per_eval": bytes_per_eval, "achieved_dt_gather_only": kern_evals_per_gpu * 4 / (kern_ms * 1e-3) / 1e9,
            "note": "algorithmic bytes per eval per SURVEY 8(d): 4 B DT voxel + 20.25 B corner-term gathers when regularization>0. `achieved` = evals x bytes / CUDA-event time of search_kernel (ONE launch per step: the rotation BnB, "
                    "every InnerBnB call and every ICP of the batch run inside it), `achieved_aggregate` = evals x bytes / step time per GPU, `achieved_dt_gather_only` counts the 4 B DT voxel alone. Only evals of calls the reference order "
                    "consumes are counted (look-ahead calls that are abandoned and corner evals are not). The 20^3 volumes are staged into shared memory by TMA (cp.async.bulk) once per pair and CTA, so the gathers are LDS and DRAM sees "
                    "staging, queue and memo traffic only: the binding limit is SM issue + the serial phases of each queue pop, not HBM (ncu on this launch: issue-active 56 %, 34 % of warp samples at a CTA barrier) -- see DESIGN.md "
                    "section 4 and profiles/. `traffic` = dram__bytes_read + dram__bytes_write of one ncu-profiled launch of the same kernel on the same 4096-pair workload at 592 CTAs (profiles/search_traffic.json; null for other workloads): queue slabs, corner memo and slot records, ~0.5 % of the algorithmic bytes"}
    # DRAM bytes of one ncu-profiled launch of the same kernel on the same workload (4096 pairs, 592 CTAs): profiles/search_traffic.json
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "search_traffic.json")))
        if int(tj.get("pairs_per_launch", 0)) == args.pairs and not args.fpfh:
            roof["traffic"] = tj.get("dram_bytes_per_launch")
    except Exception:
        pass
    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": dev_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32+f64", "data": "synthetic",
            "config": config_dict(args), "pairs_per_s": args.pairs * world * args.steps / (dev_ms * 1e-3), "ms_per_pair": dev_ms / args.steps / args.pairs,
            "wall_ms_per_step": 1e3 * wall / args.steps,
            "e2e": {"value": e2e_evals / (e2e_ms * 1e-3), "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                    "pairs_per_s": args.pairs * world * args.steps / (e2e_ms * 1e-3)},
            "gpu_launches": int(launches), "roofline": roof, "clocks": sampler.summary(),
            "rank0_last_step": {"gpu_ms": {"dt": last_tm["ms"][0], "initialize": last_tm["ms"][1], "search": last_tm["ms"][2], "icp_wave": last_tm["ms"][3]},
                                "launches": last_tm["launches"], **last_stats}}
    if world == 1 and not (args.no_cpu_baseline and args.no_per_pair):
        # the CPU legs run after every GPU measurement: the reference on the sweep sample (all cores but those of the per-pair runs) and,
        # beside it, the single-core reference on configs 1-3 (config 4 at 512^3 takes minutes of one core: --per-pair-cpu-deep)
        import multiprocessing as mp
        from oracle import pyoracle as po
        kind = "ref" if po.available("ref") else "port"
        pp, pp_async, pp_pool = None, None, None
        if not args.no_per_pair:
            cases = _pp_cases(g, synth)
            pp = per_pair_gpu(g, cases)
            cpu_cases = [c for c in cases if not c.get("deep") or args.per_pair_cpu_deep]
            pp_pool = mp.get_context("fork").Pool(len(cpu_cases))
            pp_async = pp_pool.map_async(_pp_cpu_worker, [(kind, c) for c in cpu_cases], chunksize=1)
        if not args.no_cpu_baseline:
            n = args.cpu_pairs or min(len(pairs), 16 * cores)
            sweep_cores = max(1, cores - (3 if pp_async is not None else 0))
            order = list(np.argsort([r["counters"][2] for r in res[:n]])[::-1])   # the GPU run knows every pair's cost: longest first
            cb = cpu_arm(pairs[:n], args.fpfh, sweep_cores, order)
            same = all(np.float32(e) == np.float32(r["optError"]) for e, r in zip(cb["opt_errors"], res[:n]))
            line["cpu_baseline"] = {"value": cb["value"], "unit": UNIT, "cores": sweep_cores, "kind": cb["kind"], "seconds": cb["seconds"], "per_core": cb["per_core"], "busy_fraction": cb["busy_fraction"],
                                    "sample": f"the first {n} pairs of the step's workload ({cb['evals']:.3g} evals), {sweep_cores} worker processes fed longest pair first from one queue (one reference registration per pair); "
                                              f"cores busy {100 * cb['busy_fraction']:.0f} % of the {cb['seconds']:.1f} s", "opt_error_identical_to_gpu": bool(same)}
        if pp is not None:
            cpu = pp_async.get(); pp_pool.close()
            k = 0
            for row, c in zip(pp, cases):
                if c.get("deep") and not args.per_pair_cpu_deep:
                    row.update(cpu_s_dt=None, cpu_s_register=None, speedup=None, note="reference not timed here (512^3: minutes of one core); pass --per-pair-cpu-deep")
                    continue
                tdt, treg, err = cpu[k]; k += 1
                row.update(cpu_s_dt=tdt, cpu_s_register=treg, cpu_opt_error=err, speedup=(tdt + treg) / (1e-3 * (row["gpu_ms_dt"] + row["gpu_ms_register"])),
                           speedup_register=treg / (1e-3 * row["gpu_ms_register"]), opt_error_rel_diff=abs(err - row["gpu_opt_error"]) / max(abs(err), 1e-30))
            line["per_pair"] = {"metric": "wall time per registration pair (BuildDT + Register, steady clock, no file I/O; median of 3 on the GPU, one run of the single-core reference)",
                                "cpu_kind": "reference" if kind == "ref" else "port", "rows": pp}
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
