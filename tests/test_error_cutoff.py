"""Error cutoff for screening (goicp_set_error_cutoff): a pair's search ends at the first rotation pop whose lower bound reaches its
cutoff while the reference's end test (optError - lb <= SSEThresh, jly_goicp.cpp:685) does not hold.  Everything before that pop is
the search without a cutoff, so a pair that is not cut returns exactly the uncut result, and a cut pair returns a prefix of it: the
same trace up to the new end line, counters no larger, an incumbent no better, and a lower bound lb >= cutoff on its optimum."""
import importlib
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT, golden, pair_clouds

INF = float("inf")


@pytest.fixture(scope="module")
def synth(g):
    return importlib.import_module("goicp_b200.synth")


def mixed_pairs(synth, n, seed):
    """n BO1 pairs, similar and dissimilar interleaved"""
    sim, dis = synth.bo1_pairs(n // 2, seed=seed), synth.bo1_pairs(n - n // 2, seed=seed + 1, similar=False)
    return [p for ab in zip(sim, dis) for p in ab]


def same(a, b):
    """bit-identical registrations: R, t, optError, optComp and the search counters"""
    return (np.array_equal(a["R"], b["R"]) and np.array_equal(a["t"], b["t"]) and a["optError"] == b["optError"]
            and a["optComp"] == b["optComp"] and a["counters"][:6] == b["counters"][:6])


def sse_of(params, nd):
    """SSEThresh = MSEThresh * inlierNum in float (jly_goicp.cpp:266), no trimming"""
    return np.float32(np.float32(params.MSEThresh) * np.float32(nd))


def body(trace, end="Cutoff reached"):
    """the trace lines before its end line"""
    lines = trace.splitlines()
    k = lines.index(end)
    assert len(lines) == k + 2, trace
    return lines[:k]


def is_prefix(a, b):
    return b[:len(a)] == a


def single(g, eng, pair, params, tau=None):
    reg = g.GoICP(pair["model_xyz"], pair["data_xyz"], params, engine=eng, **{k: pair[k] for k in ("model_c", "data_c", "model_fpfh", "data_fpfh")})
    reg.BuildDT(); reg.set_nd(int(pair["nd"]))
    reg.set_error_cutoff(tau)
    return reg.Register()


def test_end_lines(tmp_path):
    """CPU: the three end lines of OuterBnB as the host schedulers write them (csrc/host_search.h, plain C++), and the end kind and
    lower bound they record"""
    src = tmp_path / "ends.cpp"
    src.write_text('#include "host_search.h"\nint main() {\n'
                   '    for (int k = 1; k <= 3; k++) { SearchResult r; r.optError = 8.45388f; trace_end(r, k, 6.5f, 2.38f, 4.f);\n'
                   '                                   printf("%d %g|%s", r.endKind, r.endLb, r.trace.c_str()); }\n}\n')
    exe = str(tmp_path / "ends")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-I" + os.path.join(ROOT, "go-icp-protein-cavities_b200", "csrc"), "-o", exe, str(src), "-lm"])
    out = subprocess.run([exe], capture_output=True, text=True, check=True).stdout
    assert out == ("1 6.5|Rotation Queue Empty\nError*: 8.45388, LB: 6.5\n"
                   "2 6.5|Threshold reached\nError*: 8.45388, LB: 6.5, epsilon: 2.38\n"
                   "3 6.5|Cutoff reached\nError*: 8.45388, LB: 6.5, cutoff: 4\n")


@pytest.mark.gpu
def test_no_cutoff_changes_nothing(g, synth):
    """all cutoffs +inf, or cleared, is a run that never set one: every result and every search end bit for bit"""
    pairs = mixed_pairs(synth, 256, 5003)
    params = g.shipped_config()
    eng = g.Engine(0)
    eng.batch_upload(params, pairs)
    base = eng.batch_run()
    kind0, lb0 = eng.search_ends()
    assert set(kind0.tolist()) <= {1, 2}
    for cut in (np.full(len(pairs), INF), INF, None):
        eng.set_error_cutoff(cut)
        res = eng.batch_run()
        kind, lb = eng.search_ends()
        assert all(same(a, b) for a, b in zip(res, base)), cut
        assert np.array_equal(kind, kind0) and np.array_equal(lb, lb0), cut


@pytest.mark.gpu
def test_batch_cut_is_a_prefix(g, synth):
    """cutoff half the uncut end bound on even pairs, none on odd ones: uncut pairs are unchanged, cut pairs stop early with a
    certificate; single registrations with the same cutoff return the same result and a prefix of the uncut trace"""
    pairs = mixed_pairs(synth, 512, 7001)
    params = g.shipped_config()
    eng = g.Engine(0)
    eng.batch_upload(params, pairs)
    base = eng.batch_run()
    kind0, lb0 = eng.search_ends()
    tau = np.where(np.arange(len(pairs)) % 2 == 0, np.float32(0.5) * lb0, np.float32(INF)).astype(np.float32)
    eng.set_error_cutoff(tau)
    res = eng.batch_run()
    kind, lb = eng.search_ends()
    cut = np.flatnonzero(kind == 3)
    assert 0 < len(cut) < len(pairs)
    assert np.isfinite(tau[cut]).all()
    for i in range(len(pairs)):
        a, b = res[i], base[i]
        if kind[i] != 3:
            assert same(a, b) and kind[i] == kind0[i] and lb[i] == lb0[i], i
            continue
        assert lb[i] >= tau[i], i
        assert np.float32(a["optError"]) - lb[i] > sse_of(params, pairs[i]["nd"]), i                # :685 did not hold
        assert a["optError"] >= b["optError"], i
        assert all(x <= y for x, y in zip(a["counters"][:6], b["counters"][:6])), i
    es = g.Engine(0)
    for i in cut[:16]:
        one = single(g, es, pairs[i], params, float(tau[i]))
        k1, l1 = es.search_ends()
        assert same(one, res[i]) and k1[0] == 3 and l1[0] == lb[i], i
        full = single(g, es, pairs[i], params, None)
        assert same(full, base[i]), i
        assert is_prefix(body(one["trace"]), full["trace"].splitlines()), i


@pytest.mark.gpu
def test_cutoff_zero_cuts_at_the_root(g, synth):
    """cutoff 0: every search ends at the root pop with the incumbent of the first ICP, unless that incumbent already meets :685"""
    pairs = synth.bo1_pairs(64, seed=9001)
    params = g.shipped_config()
    eng = g.Engine(0)
    eng.batch_upload(params, pairs)
    eng.set_error_cutoff(0.0)
    res = eng.batch_run()
    kind, lb = eng.search_ends()
    es = g.Engine(0)
    for i, r in enumerate(res):
        sse = sse_of(params, pairs[i]["nd"])
        assert kind[i] == (2 if np.float32(r["optError"]) <= sse else 3), i
        assert lb[i] == 0 and r["counters"][0] == 0 and r["counters"][3] == 1, i
        one = single(g, es, pairs[i], params, 0.0)
        assert same(one, r), i
        lines = one["trace"].splitlines()
        end = 2 if lines[1].endswith("(ICP)") else 1                 # the initial error, then the first ICP's if it improved on it
        assert lines[0].endswith("(Init)") and lines[end] in ("Cutoff reached", "Threshold reached"), one["trace"]
        assert lines[end - 1].split()[1] == "%g" % r["optError"], one["trace"]
        if end == 1:
            assert np.array_equal(r["R"], np.eye(3)) and not r["t"].any(), i


CASES = {"pair2": lambda g: (g.shipped_config(), True), "deep_small": lambda g: (g.upstream_config(distTransSize=128, MSEThresh=1e-4), False)}


def check_cut(r, kind, lb, tau, sse, uncut):
    """a cut search: kind 3, lb >= tau, :685 did not hold, a prefix of the uncut trace, counters no larger"""
    assert kind == 3 and lb >= tau
    assert np.float32(r["optError"]) - lb > sse
    assert is_prefix(body(r["trace"]), uncut["trace"].splitlines())
    assert all(x <= y for x, y in zip(r["counters"][:6], uncut["counters"][:6]))


@pytest.mark.gpu
@pytest.mark.parametrize("case", sorted(CASES))
def test_every_scheduler_cuts(g, monkeypatch, case):
    """the device-resident search (where the clouds allow it), its re-run of a pair whose translation queue outgrew the kernel's
    slab, the wave scheduler and relaxed-order waves all stop with a certificate and a prefix of their own uncut trace at half the
    uncut end bound; the three exact-order runs agree bit for bit, there and at 0.95 of the end bound.  Relaxed waves test the
    cutoff only at a wave's start, so the wave that meets :685 may come first: such a run must then be the uncut one, and a
    cutoff of 0 must cut at the first wave."""
    z = golden(case)
    params, coloured = CASES[case](g)
    sse = sse_of(params, int(z["nd"]))
    reg = g.GoICP(z["model_xyz"], z["data_xyz"], params, **(pair_clouds(z) if coloured else {}))
    reg.BuildDT(); reg.set_nd(int(z["nd"]))
    full = reg.Register()
    kind0, lb0 = reg.eng.search_ends()
    assert kind0[0] in (1, 2)
    # half the end bound cuts early; 0.95 of it cuts late, after pair 2's first call that outgrows the tiny translation-queue slab
    for frac in (0.5, 0.95):
        tau = float(np.float32(frac) * lb0[0])
        reg.set_error_cutoff(tau)
        runs = {}
        # (GOICP_PERSISTENT=0 switches the handle to the wave scheduler for good: it comes last)
        for name, env in (("resident", {}), ("rerun", {"GOICP_HEAPCAP": "160"}), ("waves", {"GOICP_PERSISTENT": "0"})):
            if name == "resident":
                reg = g.GoICP(z["model_xyz"], z["data_xyz"], params, **(pair_clouds(z) if coloured else {}))
                reg.BuildDT(); reg.set_nd(int(z["nd"]))
                reg.set_error_cutoff(tau)
            with monkeypatch.context() as m:
                for k, v in env.items():
                    m.setenv(k, v)
                r = runs[name] = reg.Register()
            kind, lb = reg.eng.search_ends()
            if frac == 0.5 or kind[0] == 3:
                check_cut(r, kind[0], lb[0], tau, sse, full)
            else:   # (no pop between 0.95 of the end bound and the end)
                assert same(r, full) and r["trace"] == full["trace"], name
            if name == "rerun" and coloured and frac == 0.95:   # (the larger clouds of deep_small always run on the wave scheduler)
                assert reg.eng.stats()["search_kernel"]["pairs_rerun_by_wave_scheduler"] == 1
        for name in ("rerun", "waves"):
            assert same(runs[name], runs["resident"]) and runs[name]["trace"] == runs["resident"]["trace"], (frac, name)
    tau = float(np.float32(0.5) * lb0[0])
    reg.set_search_mode(1, 64)
    reg.set_error_cutoff(None)
    relaxed = reg.Register()
    for t in (tau, 0.0):
        reg.set_error_cutoff(t)
        r = reg.Register()
        kind, lb = reg.eng.search_ends()
        if kind[0] != 3:
            assert t > 0 and same(r, relaxed) and r["trace"] == relaxed["trace"], t
            continue
        check_cut(r, kind[0], lb[0], t, sse, relaxed)
        if t == 0:
            assert r["counters"][3] == 1 and r["counters"][0] == 0


@pytest.mark.gpu
def test_cutoff_errors(g, synth):
    """NaN, a wrong count, no problem yet, search ends before any run; a new batch upload clears the cutoffs"""
    eng = g.Engine(0)
    with pytest.raises(g.GoICPError) as e:
        eng.set_error_cutoff(1.0)
    assert e.value.status == 2
    with pytest.raises(g.GoICPError) as e:
        eng.search_ends()
    assert e.value.status == 2
    pairs = synth.bo1_pairs(8, seed=4096)
    params = g.shipped_config()
    eng.batch_upload(params, pairs)
    with pytest.raises(g.GoICPError) as e:
        eng.search_ends()
    assert e.value.status == 2
    for bad in (np.full(8, np.nan), np.array([1.0] * 7 + [np.nan]), np.ones(7), np.ones(9)):
        with pytest.raises(g.GoICPError) as e:
            eng.set_error_cutoff(bad)
        assert e.value.status == 2
    base = eng.batch_run()
    eng.set_error_cutoff(0.0)
    assert set(eng.search_ends()[0].tolist()) <= {1, 2}   # (the ends of the last run until the next one)
    cut = eng.batch_run()
    assert (eng.search_ends()[0] == 3).any() and any(not same(a, b) for a, b in zip(cut, base))
    eng.batch_upload(params, pairs)
    again = eng.batch_run()
    assert all(same(a, b) for a, b in zip(again, base)) and set(eng.search_ends()[0].tolist()) <= {1, 2}
