"""Where a batch step's time goes besides the kernels: the resident leg of bench.py for one or more builds, alternated.

    python scripts/step_overhead.py [--trees TREE[@VAR=VALUE,...] ...] [--rounds R] [--steps K] [--warmup W] [--pairs N]

Each tree is a checkout with its library built (`__graft_entry__.build()`); the default is this checkout.  `@VAR=VALUE,...` runs
the tree with those environment variables set (for instance `@GOICP_PERSISTENT=0`: the wave scheduler).  Every round runs each
tree once, in a process of its own, so that builds never share a process and the rounds interleave.  One run is bench.py's resident leg: the bench's 4096 BO1 pairs uploaded once, W warm-up steps, then K steps, each
an L2 flush and one `batch_run` between two CUDA events on the engine's stream.  Per run it prints
  - ms_per_step: the events' time per step, what the bench's headline divides by;
  - dt / initialize / search: the library's own event timings of the three phases (goicp_get_timings), mean per step;
  - gap: ms_per_step - (dt + initialize + search), the step time in which none of the three phases runs: host work, copies and
    the GPU waiting for the host;
  - host_ms: the host wall time of the step's batch_run call;
  - calls_executed / calls_used / cycles_per_pop: InnerBnB calls the search kernel ran and those the reference's order consumed,
    and CTA-cycles per translation pop inside calls (Engine.stats of the last step).
With GOICP_DEBUG set (in the environment or with @GOICP_DEBUG=1) the library's per-step search report of each run is printed
too; a tree built with `make EXTRA=-DGOICP_PHASE_TIMING` adds the cycles per pop of each phase to it.
It prints the GPU's name and power limit first and a summary of min / median / max per tree last."""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def worker(tree, steps, warmup, npairs):
    import importlib
    import torch
    sys.path.insert(0, tree)
    import __graft_entry__ as ge
    g = ge.load_package()
    synth = importlib.import_module("goicp_b200.synth")
    dev = torch.device("cuda", 0)
    stream = torch.cuda.current_stream(dev)
    eng = g.Engine(0, stream.cuda_stream)   # as bench.py: the engine on torch's current stream
    eng.set_options(1, -1, -1)
    eng.set_batch_options(-1, -1)
    params = g.shipped_config()
    pairs = synth.bo1_pairs(npairs, seed=4096)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    eng.batch_upload(params, pairs)
    for _ in range(warmup):
        flush.zero_()
        eng.batch_run()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    phase, host = [0.0, 0.0, 0.0], 0.0
    torch.cuda.synchronize(dev)
    for k in range(steps):
        flush.zero_()
        ev[k][0].record(stream)
        t0 = time.perf_counter()
        eng.batch_run()
        host += time.perf_counter() - t0
        ev[k][1].record(stream)
        ms = eng.timings()["ms"]
        for i in range(3):
            phase[i] += ms[i]
    torch.cuda.synchronize(dev)
    step = sum(a.elapsed_time(b) for a, b in ev) / steps
    dt, ini, search = (p / steps for p in phase)
    st = eng.stats()
    row = dict(tree=tree, env=os.environ.get("STEP_OVERHEAD_ENV", ""), pairs=npairs, steps=steps, ms_per_step=step, dt=dt, initialize=ini, search=search,
               gap=step - (dt + ini + search), host_ms=1e3 * host / steps, calls_executed=st["calls_executed"], calls_used=st["calls_used"],
               cycles_per_pop=st.get("search_kernel", {}).get("cycles_per_pop_in_calls"))
    print("ROW " + json.dumps(row), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--trees", nargs="+", default=[ROOT])
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--pairs", type=int, default=4096)
    ap.add_argument("--worker", help=argparse.SUPPRESS)
    a = ap.parse_args()
    if a.worker:
        return worker(a.worker, a.steps, a.warmup, a.pairs)
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    print("gpu:", q.stdout.strip().splitlines()[0] if q.returncode == 0 else "unknown (nvidia-smi failed)")
    legs = []
    for spec in a.trees:
        path, _, env = spec.partition("@")
        legs.append((spec, os.path.abspath(path), dict(kv.split("=", 1) for kv in env.split(",") if kv)))
    rows = []
    for r in range(a.rounds):
        for spec, path, env in legs:
            out = subprocess.run([sys.executable, os.path.abspath(__file__), "--worker", path, "--steps", str(a.steps), "--warmup", str(a.warmup), "--pairs", str(a.pairs)],
                                 capture_output=True, text=True, env={**os.environ, **env, "STEP_OVERHEAD_ENV": ",".join(f"{k}={v}" for k, v in env.items())})
            line = [x for x in out.stdout.splitlines() if x.startswith("ROW ")]
            if out.returncode != 0 or not line:
                print(out.stdout[-2000:], out.stderr[-4000:])
                raise SystemExit(f"worker failed on {spec}")
            if "GOICP_DEBUG" in {**os.environ, **env}:
                print(out.stderr, end="", flush=True)
            row = json.loads(line[0][4:]); row["round"] = r; row["leg"] = spec
            print(json.dumps({k: round(v, 2) if isinstance(v, float) else v for k, v in row.items()}), flush=True)
            rows.append(row)
    for spec, _, _ in legs:
        mine = [x for x in rows if x["leg"] == spec]
        summary = {}
        for k in ("ms_per_step", "dt", "initialize", "search", "gap", "host_ms"):
            v = sorted(x[k] for x in mine)
            summary[k] = dict(min=round(v[0], 2), median=round(v[len(v) // 2], 2), max=round(v[-1], 2))
        print("SUMMARY", spec, json.dumps(summary))


if __name__ == "__main__":
    main()
