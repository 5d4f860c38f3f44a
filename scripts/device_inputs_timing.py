"""Wall times of the batch upload paths and of a large BuildDT, for one or more builds of the library, alternated.

    python scripts/device_inputs_timing.py [--trees DIR ...] [--rounds R] [--reps K] [--pairs N]

Each tree is a checkout with its library built (`__graft_entry__.build()`); the default is this checkout.  Every round runs
each tree once, in a process of its own, so that builds with different kernels never share a process and the rounds
interleave.  One round of one tree times, with a host clock around work that ends in a device synchronise:
  - batch_upload of N bench-shaped BO1 pairs (synth.bo1_pairs, the bench seed) from numpy arrays;
  - batch_upload_tensors of the same pairs from packed CUDA tensors (builds that have it);
  - batch_run of the uploaded batch;
  - BuildDT of the bunny (35 947 model points) at 300^3, upstream config.
It prints the GPU's name and power limit, one JSON line per tree and round, and a summary of min / median / max per tree."""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def worker(tree, reps, npairs):
    import importlib
    import numpy as np
    import torch
    sys.path.insert(0, tree)
    import __graft_entry__ as ge
    g = ge.load_package()
    synth = importlib.import_module("goicp_b200.synth")
    dev = torch.device("cuda", 0)
    eng = g.Engine(0, torch.cuda.current_stream(dev).cuda_stream)
    params = g.shipped_config()
    pairs = synth.bo1_pairs(npairs, seed=4096)

    def timed(fn):
        fn()   # warm-up: allocations, module loads
        out = []
        for _ in range(reps):
            torch.cuda.synchronize(dev)
            t0 = time.perf_counter()
            fn()
            torch.cuda.synchronize(dev)
            out.append(1e3 * (time.perf_counter() - t0))
        return min(out)

    row = dict(tree=tree, pairs=npairs, upload_numpy_ms=timed(lambda: eng.batch_upload(params, pairs)))
    row["batch_run_ms"] = timed(eng.batch_run)
    if hasattr(eng, "batch_upload_tensors"):
        cat = lambda k, dt: torch.from_numpy(np.ascontiguousarray(np.concatenate([p[k] for p in pairs]), dtype=dt)).to(dev)
        offs = lambda k: torch.tensor(np.concatenate([[0], np.cumsum([len(p[k]) for p in pairs])]), dtype=torch.int64)
        t = dict(model_xyz=cat("model_xyz", np.float32), model_offsets=offs("model_xyz"), data_xyz=cat("data_xyz", np.float32),
                 data_offsets=offs("data_xyz"), model_c=cat("model_c", np.int32), data_c=cat("data_c", np.int32), nd=[p["nd"] for p in pairs])
        row["upload_tensors_ms"] = timed(lambda: eng.batch_upload_tensors(params, **t))
        res = eng.batch_run()
        eng.batch_upload(params, pairs)
        ref = eng.batch_run()
        row["tensors_equal_numpy"] = all(a["optError"] == b["optError"] and np.array_equal(a["R"], b["R"]) and a["counters"][:6] == b["counters"][:6]
                                         for a, b in zip(res, ref))
    z = np.load(os.path.join(tree, "tests", "golden", "bunny.npz"))
    reg = g.GoICP(z["model_xyz"], z["data_xyz"], g.upstream_config(distTransSize=300), engine=eng)
    row["bunny300_builddt_ms"] = timed(reg.BuildDT)
    print("ROW " + json.dumps(row), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--trees", nargs="+", default=[ROOT])
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--pairs", type=int, default=4096)
    ap.add_argument("--worker", help=argparse.SUPPRESS)
    a = ap.parse_args()
    if a.worker:
        return worker(a.worker, a.reps, a.pairs)
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    print("gpu:", q.stdout.strip().splitlines()[0] if q.returncode == 0 else "unknown (nvidia-smi failed)")
    rows = []
    for r in range(a.rounds):
        for tree in a.trees:
            out = subprocess.run([sys.executable, os.path.abspath(__file__), "--worker", os.path.abspath(tree), "--reps", str(a.reps), "--pairs", str(a.pairs)],
                                 capture_output=True, text=True)
            line = [x for x in out.stdout.splitlines() if x.startswith("ROW ")]
            if out.returncode != 0 or not line:
                print(out.stdout[-2000:], out.stderr[-4000:])
                raise SystemExit(f"worker failed on {tree}")
            row = json.loads(line[0][4:]); row["round"] = r
            print(json.dumps(row), flush=True)
            rows.append(row)
    for tree in a.trees:
        mine = [x for x in rows if x["tree"] == os.path.abspath(tree)]
        summary = {}
        for k in ("upload_numpy_ms", "upload_tensors_ms", "batch_run_ms", "bunny300_builddt_ms"):
            v = sorted(x[k] for x in mine if k in x)
            summary[k] = "not measured" if not v else dict(min=round(v[0], 3), median=round(v[len(v) // 2], 3), max=round(v[-1], 3))
        print("SUMMARY", tree, json.dumps(summary))


if __name__ == "__main__":
    main()
