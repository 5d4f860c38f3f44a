"""Batches registered from device-resident clouds (goicp_batch_upload_dev, Engine.batch_upload_tensors) and K1, the per-pair
preprocessing before the distance transform, which runs on the device for every input path.

The CPU part restates K1 in numpy from the reference's rules and pins the restatement to the CPU oracle.  The GPU part
(-m gpu) holds the device K1 (goicp_get_cells) to the restatement array for array, from host and from device inputs, and
holds registrations from CUDA tensors to the host-input path bit for bit."""
import ctypes as C
import importlib

import numpy as np
import pytest

from conftest import golden, pair_clouds

KNOWN_PROPS = (8204959, 30894, 15219528, 15231913, 4646984, 16741671, 7566712, 0)   # keys of jly_goicp.cpp:66-73


def k1(model_xyz, model_c, data_c, S, ef):
    """K1 as the reference computes it, for one pair: returns None for a degenerate box, "colours" for > 32 codes"""
    m = np.asarray(model_xyz, np.float32).reshape(-1, 3)
    nm = len(m)
    mc = np.zeros(nm, np.int64) if model_c is None else np.asarray(model_c, np.int64)
    dc = np.zeros(0, np.int64) if data_c is None else np.asarray(data_c, np.int64)
    # bounding cube (jly_3ddt.cpp:899-931): float extremes as doubles, every operation a separately rounded double one
    lo, hi = [float(v) for v in m.min(0)], [float(v) for v in m.max(0)]
    C3 = [(lo[a] + hi[a]) / 2 for a in range(3)]
    mn = [C3[a] - ef * (hi[a] - C3[a]) for a in range(3)]
    mxs = [C3[a] + ef * (hi[a] - C3[a]) for a in range(3)]
    side = mxs[0] - mn[0] if mxs[0] - mn[0] > mxs[1] - mn[1] else mxs[1] - mn[1]
    side = side if side > mxs[2] - mn[2] else mxs[2] - mn[2]
    box = [C3[0] - side / 2, C3[0] + side / 2, C3[1] - side / 2, C3[1] + side / 2, C3[2] - side / 2, C3[2] + side / 2]
    if not side > 0:
        return None
    scale = S / side
    # colour dictionary: ascending signed order, as the keys of std::map<int,int>
    codes = sorted(set(mc.tolist()) | set(dc.tolist()))
    if len(codes) > 32:
        return "colours"
    index = {c: k for k, c in enumerate(codes)}
    mprop = np.array([index[c] for c in mc.tolist()], np.uint8)
    dprop = np.array([index[c] for c in dc.tolist()], np.uint8)
    # seeding (:976-995): ROUND = (int)(x + 0.5), a cast that truncates toward zero; points outside [0,S) skipped (:989)
    vox = [((m[:, a].astype(np.float64) - box[2 * a]) * scale + 0.5).astype(np.int64) for a in range(3)]
    inside = np.all([(v >= 0) & (v < S) for v in vox], axis=0)
    key = (vox[2] * S + vox[1]) * S + vox[0]
    idx = np.nonzero(inside)[0]
    order = idx[np.argsort(key[idx], kind="stable")]   # ascending voxel, then ascending point index
    cell_vox, counts = np.unique(key[order], return_counts=True)
    cell_start = np.concatenate([[0], np.cumsum(counts)]).astype(np.int32)
    # colour masks (assignCellColor jly_goicp.cpp:951-969, checkProperty :1068-1092)
    nc = len(cell_vox)
    cmask, cellcol = np.zeros(nc + 1, np.uint32), np.zeros(nc, np.int32)
    for c in range(nc):
        pts = order[cell_start[c]:cell_start[c + 1]]
        cols = mc[pts]
        if (cols != cols[0]).any():
            cellcol[c] = -1
            cmask[c] = np.bitwise_or.reduce(np.uint32(1) << mprop[pts].astype(np.uint32))
        else:
            cellcol[c] = cols[0]
            cmask[c] = (1 << index[int(cols[0])]) if int(cols[0]) in KNOWN_PROPS else 0
    return dict(box=box, scale=scale, ncells=nc, cell_vox=cell_vox.astype(np.int32), cell_start=cell_start, cell_pts=order.astype(np.int32),
                cmask=cmask, cellcol=cellcol, mprop=mprop, dprop=dprop, ncolours=len(codes))


def voxel_cellc(r, S):
    """cellc on every voxel as goicp_dt_download reports it: -2 empty, -1 mixed, else the colour"""
    cc = np.full(S ** 3, -2, np.int32)
    cc[r["cell_vox"]] = r["cellcol"]
    return cc


# ---- CPU: the restatement against the CPU oracle -----------------------------------------------------------------------
@pytest.mark.parametrize("name", ["pair1", "pair2"])
def test_k1_restatement_matches_oracle(po, name):
    z = golden(name)
    o = po.Oracle("port", z["model_xyz"], z["data_xyz"], po.shipped_config(), **pair_clouds(z))
    o.build_dt()
    r = k1(z["model_xyz"], z["model_c"], z["data_c"], 20, 2.0)
    info = o.dt_info()
    assert [info[k] for k in ("xMin", "xMax", "yMin", "yMax", "zMin", "zMax", "scale")] == r["box"] + [r["scale"]]
    assert np.array_equal(o.dt_download()[3], voxel_cellc(r, 20))
    assert np.array_equal(voxel_cellc(r, 20), z["exp_dt_cellc"])


def test_k1_restatement_edge_rules():
    """the cast truncates toward zero and points outside [0,S) are dropped (expand factor 1); identical points are degenerate"""
    m = np.array([[0, 0, 0], [1, 1, 1], [0.5, 0.5, 0.5], [0.02, 0.5, 0.5]], np.float32)
    r = k1(m, None, None, 4, 1.0)
    assert r["cell_start"][-1] == 3          # the max corner lands on voxel 4 = S and is dropped
    assert 0 in r["cell_vox"]                # the min corner: (int)(0 + 0.5) = 0
    assert k1(np.ones((5, 3), np.float32), None, None, 20, 2.0) is None
    assert k1(m, np.arange(4), np.arange(100, 129), 20, 2.0) == "colours"


# ---- GPU ---------------------------------------------------------------------------------------------------------------
def synth():
    return importlib.import_module("goicp_b200.synth")


def to_tensors(torch, pairs, dev="cuda"):
    """packed ragged tensors of a list of pair dicts (the inputs of Engine.register_batch)"""
    def cat(key, dtype):
        if any(p.get(key) is None for p in pairs):
            return None
        return torch.from_numpy(np.ascontiguousarray(np.concatenate([np.asarray(p[key]) for p in pairs]), dtype=dtype)).to(dev)

    def offs(key):
        return torch.tensor(np.concatenate([[0], np.cumsum([len(np.asarray(p[key]).reshape(-1, 3)) for p in pairs])]), dtype=torch.int64)
    return dict(model_xyz=cat("model_xyz", np.float32).reshape(-1, 3), model_offsets=offs("model_xyz"),
                data_xyz=cat("data_xyz", np.float32).reshape(-1, 3), data_offsets=offs("data_xyz"),
                model_c=cat("model_c", np.int32), data_c=cat("data_c", np.int32),
                model_fpfh=cat("model_fpfh", np.float32), data_fpfh=cat("data_fpfh", np.float32),
                nd=[int(p.get("nd", 0)) for p in pairs])


def golden_pair(name, nd=True):
    z = golden(name)
    p = dict(model_xyz=z["model_xyz"], data_xyz=z["data_xyz"], nd=int(z["nd"]) if nd else 0)
    if "model_c" in z.files:
        p.update(pair_clouds(z))
    return p


def _cell_cases(g):
    s = synth()
    one = np.random.default_rng(3).uniform(-1, 1, (200, 3)).astype(np.float32)
    return {
        "bo1_256": (s.bo1_pairs(256, seed=11), g.shipped_config()),
        "pair1": ([golden_pair("pair1")], g.shipped_config()),
        "pair2": ([golden_pair("pair2")], g.shipped_config()),
        "rand_trim64": ([golden_pair("rand")], g.upstream_config(distTransSize=64, trimFraction=0.1)),
        "deep_small128": ([golden_pair("deep_small")], g.upstream_config(distTransSize=128)),
        "bunny300": ([golden_pair("bunny")], g.upstream_config(distTransSize=300)),
        "expand1": ([golden_pair("pair1"), golden_pair("pair2")], g.shipped_config(distTransExpandFactor=1.0)),
        "one_voxel": ([dict(model_xyz=one, data_xyz=one[:50], nd=0)], g.shipped_config(distTransExpandFactor=1000.0)),
    }


CELL_CASES = ["bo1_256", "pair1", "pair2", "rand_trim64", "deep_small128", "bunny300", "expand1", "one_voxel"]


@pytest.mark.gpu
@pytest.mark.parametrize("case", CELL_CASES)
@pytest.mark.parametrize("source", ["host", "device"])
def test_get_cells_equal_restatement(g, case, source):
    import torch
    pairs, params = _cell_cases(g)[case]
    eng = g.Engine(0)
    if source == "host":
        eng.batch_upload(params, pairs)
    else:
        eng.batch_upload_tensors(params, **to_tensors(torch, pairs))
    S, ef = params.distTransSize, params.distTransExpandFactor
    for k, p in enumerate(pairs):
        m = np.asarray(p["model_xyz"], np.float32).reshape(-1, 3)
        d = np.asarray(p["data_xyz"], np.float32).reshape(-1, 3)
        r = k1(m, p.get("model_c"), np.zeros(len(d), np.int32) if p.get("data_c") is None else p["data_c"], S, ef)
        got = eng.get_cells(k, len(m), len(d))
        info = got["info"]
        assert [info.xMin, info.xMax, info.yMin, info.yMax, info.zMin, info.zMax] == r["box"] and info.scale == r["scale"], (case, k)
        assert info.ncells == r["ncells"] and info.size == S
        for key in ("cell_vox", "cell_start", "cell_pts", "cmask", "mprop", "dprop"):
            assert np.array_equal(got[key], r[key]), (case, k, key)
    if case == "one_voxel":
        assert r["ncells"] == 1 and r["cell_start"][-1] == len(pairs[0]["model_xyz"])
    if case == "expand1":
        assert any(k1(p["model_xyz"], p["model_c"], p["data_c"], S, ef)["cell_start"][-1] < len(p["model_xyz"]) for p in pairs)
    eng.close()


def _same(a, b):
    for x, y in zip(a, b):
        assert np.array_equal(x["R"], y["R"]) and np.array_equal(x["t"], y["t"])
        assert x["optError"] == y["optError"] and x["optComp"] == y["optComp"]
        assert x["counters"][:6] == y["counters"][:6] and x["status"] == y["status"] == 0
    assert len(a) == len(b)


def _register_cases(g):
    s = synth()
    bo1 = s.bo1_pairs(512, seed=5)
    deep_cfg = g.upstream_config(distTransSize=128, MSEThresh=1e-4)
    return {
        "bo1_512": (bo1, g.shipped_config()),
        "bo1_512_cfpfh": (bo1, g.shipped_config(cfpfh=1, regularizationFPFH=0.000005)),
        "mixed_deep_small": ([golden_pair("deep_small")] + [dict(model_xyz=q["model_xyz"], data_xyz=q["data_xyz"], nd=q["nd"]) for q in s.bo1_pairs(3, seed=9)], deep_cfg),
    }


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["bo1_512", "bo1_512_cfpfh", "mixed_deep_small"])
def test_register_batch_tensors_equals_host(g, case):
    import torch
    pairs, params = _register_cases(g)[case]
    eng = g.Engine(0)
    ref = eng.register_batch(params, pairs)
    got = eng.register_batch_tensors(params, **to_tensors(torch, pairs))
    _same(got, ref)
    eng.close()


@pytest.mark.gpu
def test_two_runs_after_one_device_upload(g):
    import torch
    pairs = synth().bo1_pairs(64, seed=21)
    eng = g.Engine(0)
    ref = eng.register_batch(g.shipped_config(), pairs)
    eng.batch_upload_tensors(g.shipped_config(), **to_tensors(torch, pairs))
    _same(eng.batch_run(), ref)
    _same(eng.batch_run(), ref)
    eng.close()


@pytest.mark.gpu
def test_device_upload_ordered_after_torch_stream(g):
    """the clouds are written on torch's current stream behind a long kernel and passed without a synchronise"""
    import torch
    pairs = synth().bo1_pairs(128, seed=33)
    eng = g.Engine(0)
    ref = eng.register_batch(g.shipped_config(), pairs)
    t = to_tensors(torch, pairs)
    dst = {k: (torch.empty_like(v) if torch.is_tensor(v) and v.is_cuda else v) for k, v in t.items()}
    torch.cuda.synchronize()
    torch.cuda._sleep(200_000_000)   # ~0.1 s of spinning on the current stream
    for k, v in t.items():
        if torch.is_tensor(v) and v.is_cuda:
            dst[k].copy_(v, non_blocking=True)
    _same(eng.register_batch_tensors(g.shipped_config(), **dst), ref)
    eng.close()


@pytest.mark.gpu
def test_device_upload_errors(g):
    import torch
    pairs = synth().bo1_pairs(4, seed=2)
    eng = g.Engine(0)
    p = g.shipped_config()
    t = to_tensors(torch, pairs)
    for bad in (dict(model_xyz=t["model_xyz"].cpu()), dict(data_xyz=t["data_xyz"].double()), dict(model_c=t["model_c"].long()),
                dict(model_offsets=t["model_offsets"] + 1), dict(data_offsets=t["data_offsets"].cuda()),
                dict(model_fpfh=t["model_fpfh"][:, :40].contiguous()), dict(data_xyz=t["data_xyz"].t().contiguous().t())):
        with pytest.raises(ValueError):
            eng.batch_upload_tensors(p, **{**t, **bad})
    # a host pointer through the raw ABI: rejected before any launch
    m, d = pairs[0]["model_xyz"].astype(np.float32), pairs[0]["data_xyz"].astype(np.float32)
    arr = (g.PairDesc * 1)()
    arr[0] = g.PairDesc(m.ctypes.data_as(C.POINTER(C.c_float)), None, None, len(m), C.cast(C.c_void_p(t["data_xyz"].data_ptr()), C.POINTER(C.c_float)), None, None, len(d), 0)
    assert eng.L.goicp_batch_upload_dev(eng.h, C.byref(p), 1, arr) == 2
    assert b"model_xyz" in eng.L.goicp_last_error(eng.h)
    # 33 colour codes in one pair; an all-identical model cloud
    one = [dict(pairs[0])]
    one[0]["model_c"] = np.arange(len(pairs[0]["model_xyz"]), dtype=np.int32) % 33
    with pytest.raises(g.GoICPError) as e:
        eng.batch_upload_tensors(p, **to_tensors(torch, one))
    assert e.value.status == 3
    flat = [dict(pairs[0], model_xyz=np.ones((50, 3), np.float32), model_c=np.zeros(50, np.int32), model_fpfh=np.zeros((50, 41), np.float32))]
    with pytest.raises(g.GoICPError) as e:
        eng.batch_upload_tensors(p, **to_tensors(torch, flat))
    assert e.value.status == 2
    # the handle still works
    _same(eng.register_batch_tensors(p, **t), eng.register_batch(p, pairs))
    eng.close()


@pytest.mark.gpu
def test_one_pair_device_batch_dt_download(g):
    import torch
    pair = golden_pair("pair1")
    p = g.shipped_config()
    S3 = p.distTransSize ** 3
    out = []
    for source in ("host", "device"):
        eng = g.Engine(0)
        if source == "host":
            eng.batch_upload(p, [pair])
        else:
            eng.batch_upload_tensors(p, **to_tensors(torch, [pair]))
        eng.batch_run()
        dist, near, cellc = np.zeros(S3, np.float32), np.zeros((S3, 3), np.int32), np.zeros(S3, np.int32)
        eng.check(eng.L.goicp_dt_download(eng.h, dist.ctypes.data_as(C.POINTER(C.c_float)), near.ctypes.data_as(C.POINTER(C.c_int32)),
                                          cellc.ctypes.data_as(C.POINTER(C.c_int32))))
        out.append((dist, near, cellc))
        eng.close()
    z = golden("pair1")
    for a, b, ref in zip(out[0], out[1], (z["exp_dt_dist"], z["exp_dt_near"], z["exp_dt_cellc"])):
        assert np.array_equal(a, b) and np.array_equal(b, ref)
