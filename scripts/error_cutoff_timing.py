"""What an error cutoff (goicp_set_error_cutoff) saves: pairs cut, InnerBnB calls, rotation pops and step time, with no cutoff and at
several cutoffs, for one or more builds of the library, alternated.

    python scripts/error_cutoff_timing.py [--trees DIR ...] [--taus 4 8 12] [--rounds R] [--reps K] [--pairs N]

Workloads:
  - bo1: the bench's BO1 step (synth.bo1_pairs, N pairs, the bench seed), one batch_run;
  - bo1_dissimilar: N dissimilar pairs (similar=False, the same seed), one batch_run -- the sweep the reference leaves disabled;
  - pair2: cavity pair 2 of the reference's dataset on its own (tests/golden/pair2.npz), one Register.
Each tree is a checkout with its library built (`__graft_entry__.build()`); the default is this checkout.  Every round runs each tree
once, in a process of its own, so that builds never share a process and the rounds interleave.  Inside a round every repetition runs
every setting in turn (no cutoff first, then each tau), so settings alternate too; a build without goicp_set_error_cutoff runs the
no-cutoff setting only.  Step time is the device-event time around the call on the engine's stream, median over the round's
repetitions; calls and pops are the sums of counters[0] and counters[3] over the pairs.  The GPU's name and power limit are printed
first, one JSON line per tree, round, workload and setting follows, then min / median / max over rounds of every step time."""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def worker(tree, taus, reps, npairs):
    import importlib
    import numpy as np
    import torch
    sys.path.insert(0, tree)
    import __graft_entry__ as ge
    g = ge.load_package()
    synth = importlib.import_module("goicp_b200.synth")
    dev = torch.device("cuda", 0)
    stream = torch.cuda.current_stream(dev)
    eng = g.Engine(0, stream.cuda_stream)
    params = g.shipped_config()
    settings = [None] + (list(taus) if hasattr(eng, "set_error_cutoff") else [])

    def timed(fn):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize(dev)
        a.record(stream)
        out = fn()
        b.record(stream)
        torch.cuda.synchronize(dev)
        return a.elapsed_time(b), out

    def measure(name, set_cutoff, run):
        ms, last = {s: [] for s in settings}, {}
        if set_cutoff:
            set_cutoff(settings[-1])
        run()   # warm-up (module loads, allocations) with the last setting: the uncut dissimilar batch takes tens of seconds
        for rep in range(reps):
            for s in settings:
                if set_cutoff:
                    set_cutoff(s)
                t, res = timed(run)
                ms[s].append(t)
                last[s] = (res, eng.search_ends()[0] if set_cutoff else None)
        for s in settings:
            res, kinds = last[s]
            print("ROW " + json.dumps(dict(tree=tree, workload=name, cutoff=s, pairs=len(res), cut=None if kinds is None else int((kinds == 3).sum()),
                                           calls=int(sum(r["counters"][0] for r in res)), rotation_pops=int(sum(r["counters"][3] for r in res)),
                                           step_ms=float(np.median(ms[s])))), flush=True)

    for name, similar in (("bo1", True), ("bo1_dissimilar", False)):
        eng.batch_upload(params, synth.bo1_pairs(npairs, seed=4096, similar=similar))
        measure(name, eng.set_error_cutoff if len(settings) > 1 else None, eng.batch_run)
    z = np.load(os.path.join(tree, "tests", "golden", "pair2.npz"))
    reg = g.GoICP(z["model_xyz"], z["data_xyz"], params, engine=eng, model_c=z["model_c"], data_c=z["data_c"], model_fpfh=z["model_fpfh"], data_fpfh=z["data_fpfh"])
    reg.BuildDT()
    reg.set_nd(int(z["nd"]))
    measure("pair2", reg.set_error_cutoff if len(settings) > 1 else None, lambda: [reg.Register()])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--trees", nargs="+", default=[ROOT])
    ap.add_argument("--taus", nargs="+", type=float, default=[4.0, 8.0, 12.0])
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--reps", type=int, default=1)
    ap.add_argument("--pairs", type=int, default=4096)
    ap.add_argument("--worker", help=argparse.SUPPRESS)
    a = ap.parse_args()
    if a.worker:
        return worker(a.worker, a.taus, a.reps, a.pairs)
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    print("gpu:", q.stdout.strip().splitlines()[0] if q.returncode == 0 else "unknown (nvidia-smi failed)")
    rows = []
    for r in range(a.rounds):
        for tree in a.trees:
            out = subprocess.run([sys.executable, os.path.abspath(__file__), "--worker", os.path.abspath(tree), "--reps", str(a.reps), "--pairs", str(a.pairs),
                                  "--taus", *map(str, a.taus)], capture_output=True, text=True)
            lines = [x for x in out.stdout.splitlines() if x.startswith("ROW ")]
            if out.returncode != 0 or not lines:
                print(out.stdout[-2000:], out.stderr[-4000:])
                raise SystemExit(f"worker failed on {tree}")
            for line in lines:
                row = json.loads(line[4:]); row["round"] = r
                print(json.dumps(row), flush=True)
                rows.append(row)
    for tree in a.trees:
        for w in ("bo1", "bo1_dissimilar", "pair2"):
            for s in [None] + a.taus:
                v = sorted(x["step_ms"] for x in rows if x["tree"] == os.path.abspath(tree) and x["workload"] == w and x["cutoff"] == s)
                if v:
                    print("SUMMARY", json.dumps(dict(tree=tree, workload=w, cutoff=s, step_ms=dict(min=round(v[0], 3), median=round(v[len(v) // 2], 3), max=round(v[-1], 3)))))


if __name__ == "__main__":
    main()
