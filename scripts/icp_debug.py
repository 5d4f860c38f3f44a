import os, sys
import numpy as np
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import __graft_entry__ as ge
g = ge.load_package()
from oracle import pyoracle as po
z = np.load(os.path.join(ROOT, "tests/golden/pair1.npz"))
clouds = dict(model_c=z["model_c"], data_c=z["data_c"], model_fpfh=z["model_fpfh"], data_fpfh=z["data_fpfh"])
reg = g.GoICP(z["model_xyz"], z["data_xyz"], g.shipped_config(), **clouds)
reg.BuildDT(); reg.set_nd(int(z["nd"])); reg.Initialize()
o = po.Oracle("port", z["model_xyz"], z["data_xyz"], po.shipped_config(), **clouds); o.build_dt(); o.set_nd(int(z["nd"])); o.initialize()
e, R, t, corr = reg.ICP(np.eye(3), np.zeros(3)); eo, Ro, to, co = o.icp(np.eye(3), np.zeros(3))
print("err", e, eo, "dR", np.abs(R - Ro).max(), "corr eq", (corr == co).mean())
