#!/usr/bin/env python
"""Generates tests/golden/*.npz from the reference checked out at /root/reference (run in the build container only).

Inputs are the reference's own shipped data files; expected values are (a) the reference's shipped golden
outputs (output/similar1.txt, output/similar1_rescaled.txt, demo/output.txt, rot/*.mol2 RMSDs, SURVEY.md section 4) and
(b) outputs of the reference itself compiled in place (oracle/_ref/libgoicp_ref.so, oracle/Makefile).
The GPU box has no /root/reference: tests there read only these fixtures.

    python tests/golden/make_golden.py            # all fixtures (bunny/rand at 300^3 take ~2 min of CPU)
"""
import ctypes
import os
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import pyoracle as po  # noqa: E402

REF = "/root/reference"
OUT = os.path.dirname(os.path.abspath(__file__))
libc = ctypes.CDLL("libc.so.6")
libc.strtof.restype = ctypes.c_float
libc.strtof.argtypes = [ctypes.c_char_p, ctypes.c_void_p]


def strtof_all(tokens):
    return np.array([libc.strtof(t.encode(), None) for t in tokens], dtype=np.float32)


def load_xyz_txt(path):
    """upstream demo format: N then N lines 'x y z' (READMEGo-ICP.md:47-50), parsed like ifstream >> float."""
    tok = open(path).read().split()
    n = int(tok[0])
    return strtof_all(tok[1:1 + 3 * n]).reshape(n, 3)


def load_cavity(cid, pair, tmp):
    """jly_main.cpp:72-104: mol2 -> centre -> (scale applied later) ; returns raw + centred double clouds."""
    xyz, c = po.read_mol2_ref(f"{REF}/cavities/{cid}_cavity6.mol2")
    cen, mean, maxnorm = po.normalize("ref", xyz)
    tok = open(f"{REF}/cfpfh/{cid}_cavity6.cfpfh").read().split()
    fp = strtof_all(tok).reshape(-1, 41)
    assert len(fp) == len(xyz)
    return dict(raw=xyz, c=c, centred=cen, mean=mean, maxnorm=maxnorm, fpfh=fp)


def text_roundtrip(lib, xyz, c, path):
    """writeNormalizedMolCloudFile (transformation.cpp:340) then loadPointCloud (jly_main.cpp:272)."""
    a = np.ascontiguousarray(xyz, dtype=np.float64)
    cc = np.ascontiguousarray(c, dtype=np.int32)
    assert lib.ref_write_xyz(path.encode(), a.ctypes.data_as(ctypes.POINTER(ctypes.c_double)),
                             cc.ctypes.data_as(ctypes.POINTER(ctypes.c_int)), len(a)) == 0
    tok = open(path).read().split()
    n = int(tok[0])
    rows = np.array(tok[1:1 + 4 * n]).reshape(n, 4)
    return strtof_all(list(rows[:, :3].reshape(-1))).reshape(n, 3), rows[:, 3].astype(np.int64).astype(np.int32)


def run_ref(model, data, params, nd, **clouds):
    o = po.Oracle("ref", model, data, params, **clouds)
    o.build_dt()
    info = o.dt_info()
    dist, off, near, cellc = o.dt_download() if params.distTransSize <= 64 else (None, None, None, None)
    r = o.register(nd)
    o.close()
    exp = dict(R=r["R"], t=r["t"], optError=np.float32(r["optError"]), optComp=r["optComp"],
               counters=np.array(r["counters"], dtype=np.int64), trace=np.array(po.error_trace(r["trace"])),
               dt_info=np.array([info[k] for k in ("xMin", "xMax", "yMin", "yMax", "zMin", "zMax", "scale")]))
    if dist is not None:
        exp.update(dt_dist=dist, dt_off=off, dt_near=near, dt_cellc=cellc)
    print("   ", "optError", r["optError"], "comp", r["optComp"], "counters", r["counters"][:6],
          "dt %.2fs reg %.2fs" % (r["seconds_dt"], r["seconds_register"]), list(exp["trace"]))
    return exp


def protein_fixture(src, tgt, pair_exp, scale, meanS, meanT):
    """applyTransformationProtein (transformation.cpp:469) + computeRMSD (:453) inputs as arrays."""
    lib, _ = po._lib("ref")
    xyz, c = po.read_mol2_ref(f"{REF}/chains/{src}_protein.mol2")
    ali, ca = po.read_mol2_ref(f"{REF}/ref_proteins/{src}.{tgt}/aligned_{src}_protein.mol2")
    rmsd = lib.ref_rmsd(f"{REF}/ref_proteins/{src}.{tgt}/aligned_{src}_protein.mol2".encode(),
                        f"{REF}/rot/rot_{src}_protein.mol2".encode())
    rot, cr = po.read_mol2_ref(f"{REF}/rot/rot_{src}_protein.mol2")
    return dict(protein_xyz=xyz, protein_c=c, aligned_xyz=ali, aligned_c=ca, rot_xyz=rot, rmsd=np.float32(rmsd))


def make_pair(name, tgt, src, nd, tmp, fpfh_variant=False):
    print(name)
    lib, _ = po._lib("ref")
    S, T = load_cavity(src, 1, tmp), load_cavity(tgt, 1, tmp)
    scale = max(S["maxnorm"], T["maxnorm"])  # jly_main.cpp:85
    sN, tN = po.scale("ref", S["centred"], scale), po.scale("ref", T["centred"], scale)
    d_xyz, d_c = text_roundtrip(lib, sN, S["c"], os.path.join(tmp, "s.xyz"))
    m_xyz, m_c = text_roundtrip(lib, tN, T["c"], os.path.join(tmp, "t.xyz"))
    fx = dict(model_xyz=m_xyz, model_c=m_c, model_fpfh=T["fpfh"], data_xyz=d_xyz, data_c=d_c, data_fpfh=S["fpfh"],
              nd=nd, src_raw=S["raw"], tgt_raw=T["raw"], src_mean=S["mean"], tgt_mean=T["mean"],
              src_maxnorm=S["maxnorm"], tgt_maxnorm=T["maxnorm"], scale=scale, src_scaled=sN, tgt_scaled=tN)
    clouds = dict(model_c=m_c, data_c=d_c, model_fpfh=T["fpfh"], data_fpfh=S["fpfh"])
    exp = run_ref(m_xyz, d_xyz, po.shipped_config(), nd, **clouds)
    fx.update({"exp_" + k: v for k, v in exp.items()})
    # rescaled translation (transformation.cpp:410-412) via the reference's own writer
    p = os.path.join(tmp, "r.txt")
    dp = lambda a: np.ascontiguousarray(a, dtype=np.float64).ctypes.data_as(ctypes.POINTER(ctypes.c_double))
    lib.ref_rescale(p.encode(), scale, dp(T["mean"]), dp(S["mean"]), dp(exp["R"]), dp(exp["t"]), 0.0, float(exp["optError"]))
    lines = open(p).read().split("\n")
    fx["exp_rescaled_t"] = np.array([float(lines[6]), float(lines[7]), float(lines[8])])
    fx["rescaled_text"] = np.array(open(p).read())
    if fpfh_variant:
        expf = run_ref(m_xyz, d_xyz, po.shipped_config(cfpfh=1, regularizationFPFH=0.000005), nd, **clouds)
        fx.update({"expf_" + k: v for k, v in expf.items() if not k.startswith("dt_")})
        # neighbour-count term (regularizationNeighbors, jly_goicp.cpp:1200-1288)
        expn = run_ref(m_xyz, d_xyz, po.shipped_config(regularizationNeighbors=0.00001), nd, **clouds)
        fx.update({"expn_" + k: v for k, v in expn.items() if not k.startswith("dt_")})
    fx.update(protein_fixture(src, tgt, exp, scale, S["mean"], T["mean"]))
    np.savez_compressed(os.path.join(OUT, name + ".npz"), **fx)


def make_demo(name, model_f, data_f, nd, trim, sizes):
    print(name)
    m, d = load_xyz_txt(f"{REF}/demo/{model_f}"), load_xyz_txt(f"{REF}/demo/{data_f}")
    fx = dict(model_xyz=m, data_xyz=d[:max(nd, 1)] if nd else d, nd=nd, trim=np.float32(trim))
    for S in sizes:
        exp = run_ref(m, fx["data_xyz"], po.upstream_config(trimFraction=trim, distTransSize=S), nd)
        fx.update({f"exp{S}_" + k: v for k, v in exp.items()})
    np.savez_compressed(os.path.join(OUT, name + ".npz"), **fx)


def make_inclusion():
    """trimmed-error inclusion sets: the reference's own intro_select (jly_sorting.hpp:229) on residual rows of the rand demo
    clouds (trimFraction 0.1, DT 64^3) for random rotations / child translation cubes -> the values its trimmed sums run over."""
    print("inclusion")
    z = np.load(os.path.join(OUT, "rand.npz"))
    rng = np.random.default_rng(31)
    o = po.Oracle("ref", z["model_xyz"], z["data_xyz"], po.upstream_config(trimFraction=0.1, distTransSize=64))
    o.build_dt(); o.set_nd(int(z["nd"])); o.initialize()
    fx = {}
    for q, level in enumerate((-1, 0, 3)):
        v = rng.normal(size=3); v *= rng.uniform(0, np.pi) / np.linalg.norm(v)
        t = np.linalg.norm(v); k = v / t
        K = np.array([[0, -k[2], k[1]], [k[2], 0, -k[0]], [-k[1], k[0], 0]])
        R = (np.eye(3) + np.sin(t) * K + (1 - np.cos(t)) * K @ K).astype(np.float32)
        w = np.float32(0.25)
        tc = np.concatenate([rng.uniform(-0.5, 0.25, (40, 3)), np.full((40, 1), w)], 1).astype(np.float32)
        tc[:4, :3] += 3.0   # far outside the grid: many tied residuals
        firstk, resid = o.eval_inclusion(R, level, tc)
        fx.update({f"R{q}": R, f"level{q}": level, f"tc{q}": tc, f"firstk_sorted{q}": np.sort(firstk, 1), f"resid{q}": resid})
    o.close()
    np.savez_compressed(os.path.join(OUT, "rand_inclusion.npz"), **fx)


def make_inner(kind="ref"):
    """function-level values on cavity pair 2 (shipped config): weights, maxRotDis, DT3D::Distance of 2 000 seeded queries,
    InnerBnB of 6 seeded rotations at levels -1 and 1 against optError 30, and one ICP from the identity.  The inputs are the ones
    tests/test_oracle_golden.py::test_port_vs_reference_inner_calls always used, and they are stored beside the values.  `kind`
    names the implementation that produced them; it is stored as `source`."""
    print("pair2_inner", kind)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from conftest import rand_rot
    z = np.load(os.path.join(OUT, "pair2.npz"))
    o = po.Oracle(kind, z["model_xyz"], z["data_xyz"], po.shipped_config(), model_c=z["model_c"], data_c=z["data_c"],
                  model_fpfh=z["model_fpfh"], data_fpfh=z["data_fpfh"])
    o.build_dt(); o.set_nd(int(z["nd"])); o.initialize()
    rng = np.random.default_rng(1)
    q = rng.uniform(-1.5, 1.5, (2000, 3))
    Rs = np.stack([rand_rot(rng) for _ in range(6)])
    inner = [[o.inner_bnb(R, level, 30.0) for level in (-1, 1)] for R in Rs]
    e, R, t, corr = o.icp(np.eye(3), np.zeros(3))
    fx = dict(source=np.array(kind), weights=o.weights(), maxrotdis=o.maxrotdis(), q=q, dist=o.dt_distance(q)[0], R=Rs,
              levels=np.array([-1, 1], np.int32), inner_opt_error=np.float32(30.0),
              inner_err=np.array([[v[0] for v in row] for row in inner], np.float32),
              inner_tnode=np.array([[v[1] for v in row] for row in inner], np.float32),
              icp_err=np.float32(e), icp_R=R, icp_t=t, icp_corr=corr)
    o.close()
    np.savez_compressed(os.path.join(OUT, "pair2_inner.npz"), **fx)


def make_deep_small():
    """BASELINE config 4 (synthetic deep search) at a size the reference finishes in minutes: target 20 000 points on the bumpy
    sphere, source 2 000 of them moved by a random rigid motion + noise (go-icp-protein-cavities_b200/synth.py:deep_pair, seed 1241),
    DT 128^3, MSEThresh 1e-4, no trimming.  The initial ICP does not reach the optimum: 2 146 rotation nodes are expanded."""
    print("deep_small")
    import importlib.util
    spec = importlib.util.spec_from_file_location("synth", os.path.join(ROOT, "go-icp-protein-cavities_b200", "synth.py"))
    synth = importlib.util.module_from_spec(spec); spec.loader.exec_module(synth)
    p = synth.deep_pair(1241, nm=20000, nd=2000)
    fx = dict(model_xyz=p["model_xyz"], data_xyz=p["data_xyz"], nd=2000, trim=np.float32(0.0), R_true=p["R_true"], t_true=p["t_true"])
    exp = run_ref(p["model_xyz"], p["data_xyz"], po.upstream_config(distTransSize=128, MSEThresh=1e-4), 2000)
    fx.update({"exp128_" + k: v for k, v in exp.items()})
    np.savez_compressed(os.path.join(OUT, "deep_small.npz"), **fx)


if __name__ == "__main__":
    po.build("ref")
    which = sys.argv[1:] or ["pair1", "pair2", "inner", "rand", "bunny", "inclusion"]
    with tempfile.TemporaryDirectory() as tmp:
        if "pair1" in which:
            make_pair("pair1", "1eq2_6", "2x86_3", 238, tmp, fpfh_variant=True)
        if "pair2" in which:
            make_pair("pair2", "4imo_2", "2ktd_1", 247, tmp)
        if "inner" in which:
            make_inner()
        if "rand" in which:
            make_demo("rand", "model_rand.txt", "data_rand.txt", 100, 0.1, [64, 300])
        if "bunny" in which:
            make_demo("bunny", "model_bunny.txt", "data_bunny.txt", 1000, 0.0, [100, 300])
        if "inclusion" in which:
            make_inclusion()
        if "deep_small" in which:
            make_deep_small()
