"""One batch run as the host enqueues it: the "Error*:" trace recorded as values and formatted when read, the per-pair parameter
records copied to the device only when something they derive from changed, and the results converted to Python column by
column.  None of it may change a result or a trace byte."""
import ctypes as C
import importlib
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT

INF = float("inf")


def test_trace_formatted_on_read_matches_eager_text(tmp_path):
    """CPU: Trace::str (csrc/host_search.h) writes the bytes the rules used to write as they ran, for every event kind and all
    three end kinds"""
    exe = str(tmp_path / "trace_format_check")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-I" + os.path.join(ROOT, "go-icp-protein-cavities_b200", "csrc"),
                           "-o", exe, os.path.join(ROOT, "tests", "trace_format_check.cpp"), "-lm"])
    out = subprocess.run([exe, "5000"], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stdout[-3000:]
    assert out.stdout.split()[-4:] == ["cases", "5000", "mismatches", "0"], out.stdout


def test_result_columns_match_result_dict(g):
    """CPU: the column-wise conversion of a Result array gives the dicts _result_dict gives row by row: same keys, same types,
    same values"""
    rng = np.random.default_rng(7)
    n = 513
    res = (g.Result * n)()
    raw = np.frombuffer(res, np.uint8).reshape(n, -1)
    raw[:] = rng.integers(0, 256, raw.shape, dtype=np.uint8)   # every bit pattern: NaNs, infinities, denormals, negative counters
    for got, want in zip(g._result_dicts(res), [g._result_dict(r) for r in res]):
        assert list(got) == list(want)
        for k, w in want.items():
            v = got[k]
            assert type(v) is type(w), k
            if isinstance(w, np.ndarray):
                assert v.dtype == w.dtype and v.shape == w.shape and v.tobytes() == w.tobytes(), k
            elif isinstance(w, list):
                assert v == w and all(type(x) is type(y) for x, y in zip(v, w)), k
            else:
                assert v == w or (v != v and w != w), k


@pytest.fixture(scope="module")
def batch(g):
    synth = importlib.import_module("goicp_b200.synth")
    return synth.bo1_pairs(64, seed=4096)


def single(g, eng, pair, params, tau=None):
    reg = g.GoICP(pair["model_xyz"], pair["data_xyz"], params, engine=eng, **{k: pair[k] for k in ("model_c", "data_c", "model_fpfh", "data_fpfh")})
    reg.BuildDT(); reg.set_nd(int(pair["nd"]))
    reg.set_error_cutoff(tau)
    return reg.Register()


def same(a, b):
    return (np.array_equal(a["R"], b["R"]) and np.array_equal(a["t"], b["t"]) and a["optError"] == b["optError"]
            and a["optComp"] == b["optComp"] and a["counters"][:6] == b["counters"][:6])


@pytest.mark.gpu
def test_batch_trace_is_pair0_single_trace(g, batch):
    """goicp_last_trace after batch_run is the trace of registering pair 0 alone, without and with an error cutoff"""
    params = g.shipped_config()
    eng, es = g.Engine(0), g.Engine(0)
    eng.batch_upload(params, batch)
    res = eng.batch_run()
    one = single(g, es, batch[0], params)
    assert same(res[0], one)
    assert eng.last_trace() == one["trace"] and one["trace"].startswith("Error*: ") and one["trace"].endswith("\n")
    kind0, lb0 = eng.search_ends()
    tau = np.float32(0.5) * lb0   # half the uncut end bound: pair 0 is cut unless its first incumbent already meets :685
    eng.set_error_cutoff(tau)
    cut = eng.batch_run()
    kind, _ = eng.search_ends()
    one = single(g, es, batch[0], params, float(tau[0]))
    assert same(cut[0], one)
    assert eng.last_trace() == one["trace"]
    if kind[0] == 3:
        assert "Cutoff reached\n" in one["trace"]


@pytest.mark.gpu
def test_wave_scheduler_trace_is_pair0_single_trace(g, batch, monkeypatch):
    """the same with the wave scheduler (host-side OuterBnB), whose rules record the trace events themselves"""
    monkeypatch.setenv("GOICP_PERSISTENT", "0")
    params = g.shipped_config()
    eng, es = g.Engine(0), g.Engine(0)
    eng.batch_upload(params, batch)
    res = eng.batch_run()
    assert eng.stats()["waves"] > 0
    one = single(g, es, batch[0], params)
    assert same(res[0], one)
    assert eng.last_trace() == one["trace"]


@pytest.mark.gpu
def test_unchanged_inputs_skip_the_upload_and_changes_take_effect(g, batch):
    """a second batch_run with the same inputs copies no per-pair records; set_params and set_error_cutoff between runs copy
    them once and change the results as a fresh upload with those settings does"""
    params = g.shipped_config()
    eng = g.Engine(0)
    eng.batch_upload(params, batch)
    base = eng.batch_run()
    n0 = eng.pairdev_uploads()
    assert n0 >= 1
    again = eng.batch_run()
    assert eng.pairdev_uploads() == n0
    assert all(same(a, b) for a, b in zip(again, base))
    t = eng.timings()
    assert t["launches"][0] >= 1 and t["launches"][1] >= 1 and t["ms"][0] > 0 and t["ms"][1] > 0 and t["ms"][2] > 0

    looser = params.copy(MSEThresh=0.05)   # not a grid key: no new K1, only the records change
    eng.check(eng.L.goicp_set_params(eng.h, C.byref(looser)))
    res = eng.batch_run()
    assert eng.pairdev_uploads() == n0 + 1
    ref = g.Engine(0)
    ref.batch_upload(looser, batch)
    want = ref.batch_run()
    assert all(same(a, b) for a, b in zip(res, want))
    assert any(a["counters"][3] != b["counters"][3] for a, b in zip(res, base))

    eng.check(eng.L.goicp_set_params(eng.h, C.byref(params)))
    assert all(same(a, b) for a, b in zip(eng.batch_run(), base))
    n1 = eng.pairdev_uploads()
    assert n1 == n0 + 2

    kind0, lb0 = eng.search_ends()
    eng.set_error_cutoff(np.float32(0.5) * lb0)
    cut = eng.batch_run()
    kind, _ = eng.search_ends()
    assert eng.pairdev_uploads() == n1 + 1
    assert (kind == 3).any()
    assert all(same(a, b) for a, b, k in zip(cut, base, kind) if k != 3)
    eng.set_error_cutoff(None)
    assert all(same(a, b) for a, b in zip(eng.batch_run(), base))
    assert eng.pairdev_uploads() == n1 + 2
    kind, _ = eng.search_ends()
    assert np.array_equal(kind, kind0)
