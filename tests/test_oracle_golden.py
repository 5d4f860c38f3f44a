"""CPU: the oracle (plain-C restatement, oracle/goicp_oracle.c) against the reference's golden vectors -- the shipped
output files (output/similar1.txt, demo/output.txt, rot/*.mol2 RMSDs) and outputs of the reference itself compiled in
place, both frozen in tests/golden/*.npz by tests/golden/make_golden.py.  This is what pins the oracle (section 3)."""
import numpy as np
import pytest

from conftest import BACKBONE, golden, pair_clouds


def _oracle(po, z, params, kind="port"):
    return po.Oracle(kind, z["model_xyz"], z["data_xyz"], params, **pair_clouds(z))


@pytest.mark.parametrize("name", ["pair1", "pair2"])
def test_dt_bit_exact(po, name):
    """DT3D::Build: distances, 8SED offsets, emptyCells index map and cell colours equal the reference on every voxel."""
    z = golden(name)
    o = _oracle(po, z, po.shipped_config())
    o.build_dt()
    info = o.dt_info()
    assert np.array_equal([info[k] for k in ("xMin", "xMax", "yMin", "yMax", "zMin", "zMax", "scale")], z["exp_dt_info"])
    d, off, near, cc = o.dt_download()
    assert np.array_equal(d, z["exp_dt_dist"]) and np.array_equal(off, z["exp_dt_off"])
    assert np.array_equal(near, z["exp_dt_near"]) and np.array_equal(cc, z["exp_dt_cellc"])


def test_dt_rand64_bit_exact(po):
    z = golden("rand")
    o = po.Oracle("port", z["model_xyz"], z["data_xyz"], po.upstream_config(trimFraction=0.1, distTransSize=64))
    o.build_dt()
    d, off, near, cc = o.dt_download()
    assert np.array_equal(d, z["exp64_dt_dist"]) and np.array_equal(off, z["exp64_dt_off"]) and np.array_equal(near, z["exp64_dt_near"])


def test_pair1_register_golden(po):
    """output/similar1.txt: Error 8.45388, Compatibilities 133 (= 238 - 105), R/t to 7 decimals; identical node counters
    and improvement trace as the reference run."""
    z = golden("pair1")
    o = _oracle(po, z, po.shipped_config())
    r = o.register(int(z["nd"]))
    assert r["optError"] == float(z["exp_optError"]) and abs(r["optError"] - 8.45388) < 5e-6
    assert r["optComp"] == int(z["exp_optComp"]) == 238 - 133
    assert np.abs(r["R"] - z["exp_R"]).max() < 1e-12 and np.abs(r["t"] - z["exp_t"]).max() < 1e-12   # same SVD ordering as Matrix::svd
    golden_R = np.array([[0.2491547, 0.7601179, 0.6001184], [-0.7550769, -0.2355628, 0.6118569], [0.6064490, -0.6055829, 0.5152558]])
    assert np.abs(r["R"] - golden_R).max() < 1e-6
    assert r["counters"][:6] == z["exp_counters"][:6].tolist()
    assert po.error_trace(r["trace"]) == list(z["exp_trace"])


def test_pair1_fpfh_register(po):
    """cfpfh=1, regularizationFPFH=5e-6: Error 9.37283 (oracle-pinned against the reference compiled in place)"""
    z = golden("pair1")
    o = _oracle(po, z, po.shipped_config(cfpfh=1, regularizationFPFH=0.000005))
    r = o.register(int(z["nd"]))
    assert r["optError"] == float(z["expf_optError"]) and abs(r["optError"] - 9.37283) < 5e-6
    assert r["counters"][:6] == z["expf_counters"][:6].tolist()
    assert po.error_trace(r["trace"]) == list(z["expf_trace"])


def test_rand_trim_register(po):
    """trimFraction 0.1 (intro_select path), DT 64^3: same optimum as the reference (sum order differs -> tolerance)"""
    z = golden("rand")
    o = po.Oracle("port", z["model_xyz"], z["data_xyz"], po.upstream_config(trimFraction=0.1, distTransSize=64))
    r = o.register(int(z["nd"]))
    assert abs(r["optError"] - float(z["exp64_optError"])) <= 1e-5 * float(z["exp64_optError"])
    assert np.abs(r["R"] - z["exp64_R"]).max() < 1e-5 and np.abs(r["t"] - z["exp64_t"]).max() < 1e-5


def test_bunny100_register(po):
    z = golden("bunny")
    o = po.Oracle("port", z["model_xyz"], z["data_xyz"], po.upstream_config(distTransSize=100))
    r = o.register(int(z["nd"]))
    assert r["optError"] == float(z["exp100_optError"])
    assert np.abs(r["R"] - z["exp100_R"]).max() < 1e-12 and np.abs(r["t"] - z["exp100_t"]).max() < 1e-12
    assert r["counters"][:6] == z["exp100_counters"][:6].tolist()


def test_bunny300_golden_values():
    """demo/output.txt (upstream demo, DT 300^3): the frozen reference run reproduces the shipped R, t to 7 decimals"""
    z = golden("bunny")
    R = np.array([[-0.0101497, 0.0017169, 0.9999469], [-0.0041633, 0.9999896, -0.0017597], [-0.9999398, -0.0041811, -0.0101425]])
    t = np.array([0.2163900, -0.1497952, 0.0745708])
    assert np.abs(z["exp300_R"] - R).max() < 1e-7 and np.abs(z["exp300_t"] - t).max() < 1e-7
    assert abs(float(z["exp300_optError"]) - 0.145875812) < 1e-8


@pytest.mark.parametrize("name,rmsd", [("pair1", 1.736753), ("pair2", 13.929641)])
def test_transformation_golden(po, name, rmsd):
    """normalizeMolCloud / scaleCloud / rescaleCloud / applyTransformationProtein / computeRMSD against the shipped
    cavitiesN, _rescaled and rot/ artefacts (SURVEY.md section 4)."""
    z = golden(name)
    cen, mean, mx = po.normalize("port", z["src_raw"])
    assert np.allclose(mean, z["src_mean"], rtol=0, atol=1e-12) and abs(mx - float(z["src_maxnorm"])) < 1e-12
    sc = po.scale("port", cen, float(z["scale"]))
    assert np.abs(sc - z["src_scaled"]).max() < 1e-15
    lib, _ = po._lib("port")
    import ctypes as C
    dp = lambda a: np.ascontiguousarray(a, dtype=np.float64).ctypes.data_as(C.POINTER(C.c_double))
    out = np.zeros(3)
    lib.orc_rescale_translation(float(z["scale"]), dp(z["tgt_mean"]), dp(z["src_mean"]), dp(z["exp_R"]), dp(z["exp_t"]), dp(out))
    assert np.abs(out - z["exp_rescaled_t"]).max() < 5e-4   # the golden file prints 6 significant digits
    txt = str(z["rescaled_text"]).split("\n")
    R = np.array([[float(v) for v in txt[i].split()] for i in (2, 3, 4)])
    t = np.array([float(txt[i]) for i in (6, 7, 8)])
    P = np.ascontiguousarray(z["protein_xyz"], dtype=np.float64)
    rot = np.zeros_like(P)
    lib.orc_apply_rigid(dp(P), len(P), dp(R), dp(t), dp(rot))
    assert np.abs(rot[:-1] - z["rot_xyz"][:-1]).max() < 1e-6   # to_string keeps 6 decimals; the last atom is the Q6 quirk
    sel = np.isin(z["aligned_c"], BACKBONE)
    a, b = np.ascontiguousarray(z["aligned_xyz"][sel]), np.ascontiguousarray(z["rot_xyz"][sel])
    got = lib.orc_rmsd(dp(a), dp(b), len(a))
    assert abs(got - float(z["rmsd"])) < 1e-6 and abs(got - rmsd) < 1e-5


def test_port_vs_reference_inner_calls(po):
    """function-level pin on pair 2: weights / maxRotDis / Distance / InnerBnB / ICP equal tests/golden/pair2_inner.npz
    (make_golden.py: make_inner).  That file was frozen from the restatement (its `source` entry), which this test had held bit-equal
    to the reference compiled in place on these very calls; its DT distances also equal the reference's frozen DT grid (pair2.npz) at
    every in-grid query.  Where the reference is compiled (oracle/_ref), it is held to the same values."""
    z, fx = golden("pair2"), golden("pair2_inner")
    for kind in ["port"] + (["ref"] if po.available("ref") else []):
        o = _oracle(po, z, po.shipped_config(), kind)
        o.build_dt(); o.set_nd(int(z["nd"])); o.initialize()
        assert np.array_equal(o.weights(), fx["weights"]) and np.array_equal(o.maxrotdis(), fx["maxrotdis"]), kind
        assert np.array_equal(o.dt_distance(fx["q"])[0], fx["dist"]), kind
        for k, R in enumerate(fx["R"]):
            for j, level in enumerate(fx["levels"]):
                e, tn = o.inner_bnb(R, int(level), float(fx["inner_opt_error"]))
                assert e == fx["inner_err"][k, j] and (level >= 0 or np.array_equal(tn, fx["inner_tnode"][k, j])), (kind, k, int(level))
        e, R, t, corr = o.icp(np.eye(3), np.zeros(3))
        assert e == fx["icp_err"] and np.abs(R - fx["icp_R"]).max() < 1e-12 and np.abs(t - fx["icp_t"]).max() < 1e-12, kind
        assert np.array_equal(corr, fx["icp_corr"]), kind
        o.close()


def test_pair1_neighbours_term(po):
    """regularizationNeighbors = 1e-5 (assignNeighbors / nearestNeighbor / compareNeighbors, jly_goicp.cpp:1200-1288):
    the restatement equals the reference run frozen in the fixture"""
    z = golden("pair1")
    o = _oracle(po, z, po.shipped_config(regularizationNeighbors=0.00001))
    r = o.register(int(z["nd"]))
    assert r["optError"] == float(z["expn_optError"]) and r["optComp"] == int(z["expn_optComp"])
    assert r["counters"][:6] == z["expn_counters"][:6].tolist() and po.error_trace(r["trace"]) == list(z["expn_trace"])
    assert np.abs(r["R"] - z["expn_R"]).max() < 1e-12


def test_trimmed_inclusion_vs_reference_intro_select(po):
    """intro_select's contract (jly_sorting.hpp:229-313, called at jly_goicp.cpp:389): the values the reference's trimmed sums run
    over (frozen from the reference's own intro_select, tests/golden/rand_inclusion.npz) are exactly the residuals the oracle's
    inclusion mask selects; the residual rows are bit-identical"""
    z, fx = golden("rand"), golden("rand_inclusion")
    o = po.Oracle("port", z["model_xyz"], z["data_xyz"], po.upstream_config(trimFraction=0.1, distTransSize=64))
    o.build_dt(); o.set_nd(int(z["nd"])); o.initialize()
    k = o.inliernum()
    assert k == 90
    for q in range(3):
        mask, resid = o.eval_inclusion(fx[f"R{q}"], int(fx[f"level{q}"]), fx[f"tc{q}"])
        assert np.array_equal(resid, fx[f"resid{q}"])
        assert (mask.sum(1) == k).all()
        sel = np.sort(np.where(mask.astype(bool), resid, np.inf), 1)[:, :k]
        assert np.array_equal(sel, fx[f"firstk_sorted{q}"])
