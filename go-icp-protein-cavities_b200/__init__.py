"""goicp_b200 -- host-side Python mirror of the reference's C++ surface over the C ABI of libgoicp_b200.so.

The compiled reference has no Python API; its surface is the C++ classes ``GoICP`` (jly_goicp.h:112-218), ``DT3D``
(jly_3ddt.h:123-139) and ``Transformation`` (transformation.hpp:38-68).  This module keeps their names, field names and
call order (``BuildDT`` -> ``Register``; ``Initialize``/``InnerBnB``/``ICP`` exposed for parity tests) so that tests read
like a harness around the reference, and forwards every numeric call to the CUDA library through ctypes
(include/goicp_b200.h).  There is no CPU fallback: if the library or a CUDA device is missing, construction raises.

The package directory name contains hyphens (repo convention); load it with ``load_package()`` from
``__graft_entry__`` or via importlib (tests/conftest.py does this) under the module name ``goicp_b200``.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("GOICP_LIB") or os.path.join(_HERE, "libgoicp_b200.so")   # GOICP_LIB: development A/B builds


class GoICPError(RuntimeError):
    def __init__(self, status, msg):
        super().__init__(f"goicp status {status}: {msg}")
        self.status = status


class Params(C.Structure):
    """config.txt keys (readConfig, jly_main.cpp:231-270) = goicp_params."""
    _fields_ = [("MSEThresh", C.c_float),
                ("rotMinX", C.c_float), ("rotMinY", C.c_float), ("rotMinZ", C.c_float), ("rotWidth", C.c_float),
                ("transMinX", C.c_float), ("transMinY", C.c_float), ("transMinZ", C.c_float), ("transWidth", C.c_float),
                ("trimFraction", C.c_float),
                ("regularization", C.c_float), ("regularizationNeighbors", C.c_float), ("regularizationFPFH", C.c_float),
                ("cfpfh", C.c_int32), ("norm", C.c_int32), ("ponderation", C.c_int32),
                ("distTransSize", C.c_int32),
                ("distTransExpandFactor", C.c_double)]

    def copy(self, **kw):
        p = Params.from_buffer_copy(bytes(self))
        for k, v in kw.items():
            setattr(p, k, v)
        return p


class DTInfo(C.Structure):
    _fields_ = [("xMin", C.c_double), ("xMax", C.c_double), ("yMin", C.c_double), ("yMax", C.c_double),
                ("zMin", C.c_double), ("zMax", C.c_double), ("scale", C.c_double), ("size", C.c_int32), ("ncells", C.c_int32)]


class Result(C.Structure):
    _fields_ = [("R", C.c_double * 9), ("t", C.c_double * 3), ("optError", C.c_float), ("optComp", C.c_int32),
                ("counters", C.c_int64 * 8), ("seconds_dt", C.c_double), ("seconds_register", C.c_double),
                ("gpu_ms_dt", C.c_float), ("gpu_ms_bnb", C.c_float), ("gpu_ms_icp", C.c_float), ("status", C.c_int32)]


class PairDesc(C.Structure):
    _fields_ = [("model_xyz", C.POINTER(C.c_float)), ("model_c", C.POINTER(C.c_int32)), ("model_fpfh", C.POINTER(C.c_float)), ("Nm", C.c_int32),
                ("data_xyz", C.POINTER(C.c_float)), ("data_c", C.POINTER(C.c_int32)), ("data_fpfh", C.POINTER(C.c_float)), ("NdAll", C.c_int32),
                ("Nd", C.c_int32)]


# every symbol include/goicp_b200.h declares (tests/test_abi.py checks the header against this list and the .so)
ABI_SYMBOLS = [
    "goicp_version", "goicp_last_error", "goicp_params_default", "goicp_create", "goicp_destroy",
    "goicp_set_model", "goicp_set_data", "goicp_set_params", "goicp_build_dt", "goicp_build_dt_replay", "goicp_dt_upload",
    "goicp_dt_download", "goicp_dt_distance", "goicp_set_nd", "goicp_initialize", "goicp_get_weights", "goicp_get_maxrotdis",
    "goicp_get_thresholds", "goicp_eval_bounds", "goicp_eval_inclusion", "goicp_inner_bnb", "goicp_icp", "goicp_register", "goicp_outer_bnb", "goicp_last_trace",
    "goicp_set_options", "goicp_set_search_mode", "goicp_register_batch", "goicp_batch_upload", "goicp_batch_upload_dev", "goicp_batch_run",
    "goicp_get_cells", "goicp_get_timings",
    "goicp_set_batch_options", "goicp_get_stats", "goicp_set_frontier_sharding", "goicp_test_exchange",
    "goicp_normalize_cloud", "goicp_scale_cloud", "goicp_rescale_translation", "goicp_apply_rigid", "goicp_rmsd",
]

ALLGATHER_FN = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p)

_lib = None


def lib():
    """Loads libgoicp_b200.so (built in-tree by csrc/Makefile / __graft_entry__.build()).  Fails loudly when missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise FileNotFoundError(f"{LIB_PATH} not built: run `python -c 'import __graft_entry__ as g; g.build()'` (no CPU fallback exists)")
    L = C.CDLL(LIB_PATH)
    vp, fp, ip, dp = C.c_void_p, C.POINTER(C.c_float), C.POINTER(C.c_int32), C.POINTER(C.c_double)
    L.goicp_version.restype = C.c_char_p
    L.goicp_last_error.restype = C.c_char_p
    L.goicp_last_error.argtypes = [vp]
    L.goicp_last_trace.restype = C.c_char_p
    L.goicp_last_trace.argtypes = [vp]
    L.goicp_params_default.argtypes = [C.POINTER(Params)]
    L.goicp_create.argtypes = [C.POINTER(vp), C.c_int, vp]
    L.goicp_destroy.argtypes = [vp]
    L.goicp_destroy.restype = None
    L.goicp_set_model.argtypes = [vp, fp, ip, fp, C.c_int32]
    L.goicp_set_data.argtypes = [vp, fp, ip, fp, C.c_int32]
    L.goicp_set_params.argtypes = [vp, C.POINTER(Params)]
    L.goicp_build_dt.argtypes = [vp, C.POINTER(DTInfo)]
    L.goicp_build_dt_replay.argtypes = [vp, C.POINTER(DTInfo)]
    L.goicp_dt_upload.argtypes = [vp, fp, ip]
    L.goicp_dt_download.argtypes = [vp, fp, ip, ip]
    L.goicp_dt_distance.argtypes = [vp, dp, C.c_int32, fp, ip]
    L.goicp_set_nd.argtypes = [vp, C.c_int32]
    L.goicp_initialize.argtypes = [vp]
    L.goicp_get_weights.argtypes = [vp, fp]
    L.goicp_get_maxrotdis.argtypes = [vp, fp]
    L.goicp_get_thresholds.argtypes = [vp, fp, ip]
    L.goicp_eval_bounds.argtypes = [vp, fp, ip, C.c_int32, fp, ip, C.c_int32, fp, fp, ip, ip]
    L.goicp_eval_inclusion.argtypes = [vp, fp, C.c_int32, fp, C.c_int32, C.POINTER(C.c_uint8), fp]
    L.goicp_inner_bnb.argtypes = [vp, fp, ip, fp, C.c_int32, fp, fp, C.POINTER(C.c_int64)]
    L.goicp_icp.argtypes = [vp, dp, dp, fp, ip]
    L.goicp_register.argtypes = [vp, C.POINTER(Result)]
    L.goicp_outer_bnb.argtypes = [vp, C.POINTER(Result)]
    L.goicp_set_options.argtypes = [vp, C.c_int32, C.c_int32, C.c_int32]
    L.goicp_set_search_mode.argtypes = [vp, C.c_int32, C.c_int32]
    L.goicp_register_batch.argtypes = [vp, C.POINTER(Params), C.c_int32, C.POINTER(PairDesc), C.POINTER(Result)]
    L.goicp_batch_upload.argtypes = [vp, C.POINTER(Params), C.c_int32, C.POINTER(PairDesc)]
    L.goicp_batch_upload_dev.argtypes = [vp, C.POINTER(Params), C.c_int32, C.POINTER(PairDesc)]
    L.goicp_batch_run.argtypes = [vp, C.POINTER(Result)]
    u8p = C.POINTER(C.c_uint8)
    L.goicp_get_cells.argtypes = [vp, C.c_int32, ip, ip, ip, C.POINTER(C.c_uint32), u8p, u8p, C.POINTER(DTInfo)]
    L.goicp_get_timings.argtypes = [vp, fp, C.POINTER(C.c_int64)]
    L.goicp_set_batch_options.argtypes = [vp, C.c_int32, C.c_int32]
    L.goicp_get_stats.argtypes = [vp, dp]
    L.goicp_set_frontier_sharding.argtypes = [vp, C.c_int32, C.c_int32, ALLGATHER_FN, vp]
    L.goicp_test_exchange.argtypes = [vp, vp, vp, C.c_int64]
    L.goicp_normalize_cloud.argtypes = [vp, dp, C.c_int32, dp, dp]
    L.goicp_scale_cloud.argtypes = [vp, dp, C.c_int32, C.c_double]
    L.goicp_rescale_translation.argtypes = [vp, C.c_double, dp, dp, dp, dp, dp]
    L.goicp_apply_rigid.argtypes = [vp, dp, C.c_int32, dp, dp, dp]
    L.goicp_rmsd.argtypes = [vp, dp, dp, C.c_int32, fp]
    _lib = L
    return L


def shipped_config(**kw):
    """The shipped config.txt (config.txt:4-53)."""
    p = Params()
    lib().goicp_params_default(C.byref(p))
    for k, v in kw.items():
        setattr(p, k, v)
    return p


def upstream_config(**kw):
    """The upstream Go-ICP demo config (READMEGo-ICP.md:33-41): MSE 1e-3, DT 300^3, no fork terms."""
    p = Params(0.001, -3.1416, -3.1416, -3.1416, 6.2832, -0.5, -0.5, -0.5, 1.0, 0.0, 0.0, 0.0, 0.0, 0, 2, 0, 300, 2.0)
    for k, v in kw.items():
        setattr(p, k, v)
    return p


def _f32(a):
    return np.ascontiguousarray(a, dtype=np.float32)


def _i32(a):
    return np.ascontiguousarray(a, dtype=np.int32)


def _f64(a):
    return np.ascontiguousarray(a, dtype=np.float64)


def _p(a, t):
    return None if a is None else a.ctypes.data_as(C.POINTER(t))


class Engine:
    """One goicp_handle (one CUDA device + stream)."""

    def __init__(self, device=0, stream=None):
        self.L = lib()
        self.h = C.c_void_p()
        st = self.L.goicp_create(C.byref(self.h), device, stream)
        if st != 0:
            raise GoICPError(st, self.L.goicp_last_error(None).decode())

    def check(self, st):
        if st != 0:
            raise GoICPError(st, self.L.goicp_last_error(self.h).decode())

    def close(self):
        if getattr(self, "h", None):
            self.L.goicp_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def timings(self):
        ms = (C.c_float * 5)()
        ln = (C.c_int64 * 5)()
        self.check(self.L.goicp_get_timings(self.h, ms, ln))
        return dict(ms=list(ms), launches=list(ln))

    def set_frontier_sharding(self, rank, world, device=None):
        """Shard the InnerBnB calls of every wave of ONE registration over `world` ranks (torch.distributed must be
        initialised): results are all-gathered once per wave (NCCL when `device` is a cuda device, else gloo)."""
        import torch
        import torch.distributed as dist

        def _allgather(send, recv, nbytes, user):
            try:
                src = np.ctypeslib.as_array(C.cast(send, C.POINTER(C.c_uint8)), shape=(nbytes,))
                dst = np.ctypeslib.as_array(C.cast(recv, C.POINTER(C.c_uint8)), shape=(nbytes * world,))
                t = torch.from_numpy(src.copy())
                if device is not None:
                    t = t.to(device)
                out = torch.empty(nbytes * world, dtype=torch.uint8, device=t.device)
                dist.all_gather_into_tensor(out, t)
                dst[:] = out.cpu().numpy()
                return 0
            except Exception as exc:  # noqa: BLE001 - reported through the status code
                print("all-gather callback failed:", exc)
                return 1
        self._ag = ALLGATHER_FN(_allgather)   # keep the callback alive
        self.check(self.L.goicp_set_frontier_sharding(self.h, rank, world, self._ag, None))

    def stats(self):
        o = (C.c_double * 16)()
        self.check(self.L.goicp_get_stats(self.h, o))
        d = dict(waves=int(o[0]), calls_executed=int(o[1]), calls_used=int(o[2]), host_worker_threads=int(o[3]), host_seconds=o[4])
        if o[13] > 0:   # device-resident search (k_search.cu)
            d["search_kernel"] = dict(ctas=int(o[13]), calls=int(o[8]), pops=int(o[9]), cycles_per_pop_in_calls=o[10] / max(o[9], 1.0), corner_misses_per_pop=o[11] / max(o[9], 1.0),
                                      cta_cycles_total=o[15], cta_cycles_in_calls=o[10], cta_cycles_scheduling_and_idle=o[12], pairs_rerun_by_wave_scheduler=int(o[14]))
        else:           # wave scheduler
            d["host_thread_seconds"] = dict(build_requests=o[5], enqueue=o[6], wait=o[7])
        return d

    def set_options(self, exact_sums=-1, spec_width=-1, use_dt_replay=-1):
        self.check(self.L.goicp_set_options(self.h, exact_sums, spec_width, use_dt_replay))

    def set_search_mode(self, relaxed_order=-1, wave_nodes=-1):
        """single registrations: 0 = the reference's visitation order (default), 1 = relaxed-order frontier waves of `wave_nodes` rotation nodes"""
        self.check(self.L.goicp_set_search_mode(self.h, relaxed_order, wave_nodes))

    def set_batch_options(self, groups=-1, slots=-1):
        self.check(self.L.goicp_set_batch_options(self.h, groups, slots))

    # ---- batch of pairs (bo1_GoICP.py:40-54) ----
    def _descs(self, pairs):
        keep, arr = [], (PairDesc * len(pairs))()
        for i, pr in enumerate(pairs):
            m, d = _f32(pr["model_xyz"]).reshape(-1, 3), _f32(pr["data_xyz"]).reshape(-1, 3)
            mc = None if pr.get("model_c") is None else _i32(pr["model_c"])
            dc = None if pr.get("data_c") is None else _i32(pr["data_c"])
            mf = None if pr.get("model_fpfh") is None else _f32(pr["model_fpfh"])
            df = None if pr.get("data_fpfh") is None else _f32(pr["data_fpfh"])
            keep += [m, d, mc, dc, mf, df]
            arr[i] = PairDesc(_p(m, C.c_float), _p(mc, C.c_int32), _p(mf, C.c_float), len(m),
                              _p(d, C.c_float), _p(dc, C.c_int32), _p(df, C.c_float), len(d), int(pr.get("nd", 0)))
        return arr, keep

    def make_descs(self, pairs):
        """goicp_pair_desc array over the callers' host buffers (kept alive by the returned object)"""
        arr, keep = self._descs(pairs)
        return dict(arr=arr, keep=keep, n=len(pairs))

    def register_batch_descs(self, params, descs):
        """goicp_register_batch on a prepared descriptor array: host buffers in, results out"""
        res = (Result * descs["n"])()
        self.check(self.L.goicp_register_batch(self.h, C.byref(params), descs["n"], descs["arr"], res))
        return res

    def batch_upload(self, params, pairs):
        arr, keep = self._descs(pairs)
        self._npairs = len(pairs)
        self.check(self.L.goicp_batch_upload(self.h, C.byref(params), len(pairs), arr))

    def batch_run(self):
        res = (Result * self._npairs)()
        self.check(self.L.goicp_batch_run(self.h, res))
        return [_result_dict(r) for r in res]

    def register_batch(self, params, pairs):
        arr, keep = self._descs(pairs)
        res = (Result * len(pairs))()
        self.check(self.L.goicp_register_batch(self.h, C.byref(params), len(pairs), arr, res))
        return [_result_dict(r) for r in res]

    def batch_upload_tensors(self, params, model_xyz, model_offsets, data_xyz, data_offsets, model_c=None, data_c=None,
                             model_fpfh=None, data_fpfh=None, nd=None):
        """goicp_batch_upload_dev from packed ragged CUDA tensors: pair k's model is model_xyz[model_offsets[k]:model_offsets[k+1]]
        (float32 [sum Nm, 3]), likewise the data cloud; colours int32 [sum N], c-FPFH rows float32 [sum N, 41]; offsets are CPU
        int64 [P+1] (the sizes are needed on the host); nd: per-pair NdDownsampled (0 = all) or None.  The clouds are read
        after the work already queued on torch's current stream of their device; batch_run() follows."""
        import torch
        dev = _cuda_tensor(torch, model_xyz, "model_xyz", torch.float32, (None, 3)).device
        _cuda_tensor(torch, data_xyz, "data_xyz", torch.float32, (None, 3), dev)
        mo = _offsets(torch, model_offsets, model_xyz.shape[0], "model_offsets")
        do = _offsets(torch, data_offsets, data_xyz.shape[0], "data_offsets")
        if len(mo) != len(do):
            raise ValueError("model_offsets and data_offsets describe different numbers of pairs")
        npairs = len(mo) - 1
        tm = dict(model_c=(model_c, torch.int32, (int(mo[-1]),)), model_fpfh=(model_fpfh, torch.float32, (int(mo[-1]), 41)),
                  data_c=(data_c, torch.int32, (int(do[-1]),)), data_fpfh=(data_fpfh, torch.float32, (int(do[-1]), 41)))
        for name, (t, dt, shape) in tm.items():
            if t is not None:
                _cuda_tensor(torch, t, name, dt, shape, dev)
        if nd is not None and len(nd) != npairs:
            raise ValueError(f"nd has {len(nd)} entries for {npairs} pairs")
        arr = (PairDesc * npairs)()

        def at(t, off, row):
            return None if t is None else C.cast(C.c_void_p(t.data_ptr() + int(off) * row), C.POINTER(C.c_float if t.dtype == torch.float32 else C.c_int32))
        for k in range(npairs):
            arr[k] = PairDesc(at(model_xyz, mo[k], 12), at(model_c, mo[k], 4), at(model_fpfh, mo[k], 164), int(mo[k + 1] - mo[k]),
                              at(data_xyz, do[k], 12), at(data_c, do[k], 4), at(data_fpfh, do[k], 164), int(do[k + 1] - do[k]),
                              0 if nd is None else int(nd[k]))
        torch.cuda.current_stream(dev).synchronize()   # the clouds may still be written on torch's stream
        self._npairs = npairs
        self.check(self.L.goicp_batch_upload_dev(self.h, C.byref(params), npairs, arr))

    def register_batch_tensors(self, params, *args, **kw):
        """batch_upload_tensors + batch_run: the per-pair result dicts of register_batch"""
        self.batch_upload_tensors(params, *args, **kw)
        return self.batch_run()

    def get_cells(self, pair, nm, ndall):
        """goicp_get_cells: the cell lists, colour masks and colour indices the grid of `pair` (nm model and ndall data points)
        was built from"""
        info = DTInfo()
        self.check(self.L.goicp_get_cells(self.h, pair, None, None, None, None, None, None, C.byref(info)))
        nc = info.ncells
        start = np.zeros(nc + 1, np.int32)
        self.check(self.L.goicp_get_cells(self.h, pair, None, _p(start, C.c_int32), None, None, None, None, None))
        vox, pts, cmask = np.zeros(nc, np.int32), np.zeros(int(start[-1]), np.int32), np.zeros(nc + 1, np.uint32)
        mprop, dprop = np.zeros(nm, np.uint8), np.zeros(ndall, np.uint8)
        self.check(self.L.goicp_get_cells(self.h, pair, _p(vox, C.c_int32), None, _p(pts, C.c_int32), _p(cmask, C.c_uint32),
                                          _p(mprop, C.c_uint8), _p(dprop, C.c_uint8), None))
        return dict(cell_vox=vox, cell_start=start, cell_pts=pts, cmask=cmask, mprop=mprop, dprop=dprop, info=info)

    # ---- Transformation (transformation.cpp) ----
    def normalizeMolCloud(self, xyz):
        """:311 -- returns (centred cloud, mean, max norm)"""
        a = _f64(xyz).reshape(-1, 3).copy()
        mean, mx = np.zeros(3), C.c_double()
        self.check(self.L.goicp_normalize_cloud(self.h, _p(a, C.c_double), len(a), _p(mean, C.c_double), C.byref(mx)))
        return a, mean, mx.value

    def scaleCloud(self, xyz, scale):
        a = _f64(xyz).reshape(-1, 3).copy()
        self.check(self.L.goicp_scale_cloud(self.h, _p(a, C.c_double), len(a), scale))
        return a

    def rescaleCloud(self, scale, meanT, meanS, R, t):
        """:403-412 -- the rescaled translation"""
        out = np.zeros(3)
        self.check(self.L.goicp_rescale_translation(self.h, scale, _p(_f64(meanT), C.c_double), _p(_f64(meanS), C.c_double),
                                                    _p(_f64(R).reshape(9), C.c_double), _p(_f64(t), C.c_double), _p(out, C.c_double)))
        return out

    def applyTransformationProtein(self, xyz, R, t):
        a = _f64(xyz).reshape(-1, 3)
        out = np.zeros_like(a)
        self.check(self.L.goicp_apply_rigid(self.h, _p(a, C.c_double), len(a), _p(_f64(R).reshape(9), C.c_double), _p(_f64(t), C.c_double), _p(out, C.c_double)))
        return out

    def computeRMSD(self, a, b):
        a, b = _f64(a).reshape(-1, 3), _f64(b).reshape(-1, 3)
        out = C.c_float()
        self.check(self.L.goicp_rmsd(self.h, _p(a, C.c_double), _p(b, C.c_double), len(a), C.byref(out)))
        return float(out.value)


def _cuda_tensor(torch, t, name, dtype, shape, device=None):
    """t must be a contiguous CUDA tensor of `dtype` with `shape` (None: any length), on `device` when given"""
    if not torch.is_tensor(t) or not t.is_cuda:
        raise ValueError(f"{name} must be a CUDA tensor")
    if t.dtype != dtype:
        raise ValueError(f"{name} must be {dtype}, not {t.dtype}")
    if not t.is_contiguous():
        raise ValueError(f"{name} must be contiguous")
    if t.dim() != len(shape) or any(w is not None and w != v for w, v in zip(shape, t.shape)):
        raise ValueError(f"{name} has shape {tuple(t.shape)}, expected {tuple('N' if w is None else w for w in shape)}")
    if device is not None and t.device != device:
        raise ValueError(f"{name} is on {t.device}, the clouds on {device}")
    return t


def _offsets(torch, o, n, name):
    """CPU int64 [P+1] offsets into an array of n rows: 0 first, n last, every pair non-empty"""
    if not torch.is_tensor(o) or o.is_cuda or o.dtype != torch.int64 or o.dim() != 1 or len(o) < 2:
        raise ValueError(f"{name} must be a CPU int64 tensor of P+1 offsets")
    a = o.numpy()
    if a[0] != 0 or a[-1] != n or (np.diff(a) < 1).any():
        raise ValueError(f"{name} must rise strictly from 0 to {n}")
    if np.diff(a).max() >= 2 ** 31:
        raise ValueError(f"{name}: a cloud has 2^31 points or more")
    return a


def _result_dict(r):
    return dict(R=np.array(r.R).reshape(3, 3), t=np.array(r.t), optError=float(np.float32(r.optError)), optComp=int(r.optComp),
                counters=list(r.counters), seconds_dt=r.seconds_dt, seconds_register=r.seconds_register,
                gpu_ms_dt=r.gpu_ms_dt, gpu_ms_bnb=r.gpu_ms_bnb, gpu_ms_icp=r.gpu_ms_icp, status=int(r.status))


class GoICP:
    """Mirror of class GoICP (jly_goicp.h:112-218): set pModel/pData + config fields, BuildDT(), Register()."""

    def __init__(self, model_xyz, data_xyz, params, model_c=None, data_c=None, model_fpfh=None, data_fpfh=None, device=0, engine=None):
        self.eng = engine or Engine(device)
        self.L, self.h = self.eng.L, self.eng.h
        self.pModel, self.pData = _f32(model_xyz).reshape(-1, 3), _f32(data_xyz).reshape(-1, 3)
        self.Nm, self.Nd = len(self.pModel), len(self.pData)
        self.params = params
        mc = None if model_c is None else _i32(model_c)
        dc = None if data_c is None else _i32(data_c)
        mf = None if model_fpfh is None else _f32(model_fpfh)
        df = None if data_fpfh is None else _f32(data_fpfh)
        self.eng.check(self.L.goicp_set_params(self.h, C.byref(params)))
        self.eng.check(self.L.goicp_set_model(self.h, _p(self.pModel, C.c_float), _p(mc, C.c_int32), _p(mf, C.c_float), self.Nm))
        self.eng.check(self.L.goicp_set_data(self.h, _p(self.pData, C.c_float), _p(dc, C.c_int32), _p(df, C.c_float), self.Nd))
        self.dt = None
        self.optError, self.optR, self.optT, self.optComp = None, np.eye(3), np.zeros(3), 0

    def set_params(self, params):
        self.params = params
        self.eng.check(self.L.goicp_set_params(self.h, C.byref(params)))

    def set_search_mode(self, relaxed_order=-1, wave_nodes=-1):
        self.eng.set_search_mode(relaxed_order, wave_nodes)

    def set_options(self, exact_sums=-1, spec_width=-1, use_dt_replay=-1):
        self.eng.check(self.L.goicp_set_options(self.h, exact_sums, spec_width, use_dt_replay))

    def BuildDT(self, replay=None):
        """GoICP::BuildDT (jly_goicp.cpp:79)"""
        info = DTInfo()
        if replay:
            self.eng.check(self.L.goicp_build_dt_replay(self.h, C.byref(info)))
        else:
            self.eng.check(self.L.goicp_build_dt(self.h, C.byref(info)))
        self.dt = info
        return info

    def set_nd(self, nd):
        """`goicp.Nd = NdDownsampled` (jly_main.cpp:114-117)"""
        self.Nd = nd
        self.eng.check(self.L.goicp_set_nd(self.h, nd))

    def dt_download(self):
        S3 = self.params.distTransSize ** 3
        dist, near, cellc = np.zeros(S3, np.float32), np.zeros((S3, 3), np.int32), np.zeros(S3, np.int32)
        self.eng.check(self.L.goicp_dt_download(self.h, _p(dist, C.c_float), _p(near, C.c_int32), _p(cellc, C.c_int32)))
        return dist, near, cellc

    def dt_upload(self, dist=None, nearest=None):
        d = None if dist is None else _f32(dist)
        n = None if nearest is None else _i32(nearest)
        self.eng.check(self.L.goicp_dt_upload(self.h, _p(d, C.c_float), _p(n, C.c_int32)))

    def Distance(self, xyz):
        """DT3D::Distance (jly_3ddt.cpp:1139), batched"""
        a = _f64(xyz).reshape(-1, 3)
        out, cell = np.zeros(len(a), np.float32), np.zeros((len(a), 3), np.int32)
        self.eng.check(self.L.goicp_dt_distance(self.h, _p(a, C.c_double), len(a), _p(out, C.c_float), _p(cell, C.c_int32)))
        return out, cell

    def Initialize(self):
        self.eng.check(self.L.goicp_initialize(self.h))

    def weights(self):
        w = np.zeros(self.Nd, np.float32)
        self.eng.check(self.L.goicp_get_weights(self.h, _p(w, C.c_float)))
        return w

    def maxRotDis(self):
        w = np.zeros((20, self.Nd), np.float32)
        self.eng.check(self.L.goicp_get_maxrotdis(self.h, _p(w, C.c_float)))
        return w

    def thresholds(self):
        sse, inl = C.c_float(), C.c_int32()
        self.eng.check(self.L.goicp_get_thresholds(self.h, C.byref(sse), C.byref(inl)))
        return float(sse.value), int(inl.value)

    def eval_bounds(self, R, level, tcubes, rot_of=None):
        R = _f32(R).reshape(-1, 9)
        level = _i32(np.atleast_1d(level))
        tc = _f32(tcubes).reshape(-1, 4)
        n = len(tc)
        ro = _i32(np.zeros(n) if rot_of is None else rot_of)
        ub, lb = np.zeros(n, np.float32), np.zeros(n, np.float32)
        inc, fp = np.zeros((n, 2), np.int32), np.zeros((n, 2), np.int32)
        self.eng.check(self.L.goicp_eval_bounds(self.h, _p(R, C.c_float), _p(level, C.c_int32), len(R), _p(tc, C.c_float), _p(ro, C.c_int32), n,
                                                _p(ub, C.c_float), _p(lb, C.c_float), _p(inc, C.c_int32), _p(fp, C.c_int32)))
        return ub, lb, inc, fp

    def eval_inclusion(self, R, level, tcubes):
        """per-cube point-inclusion masks of the trimmed error (intro_select's contract) + the residual rows: (mask[n,Nd] uint8, resid[n,Nd])"""
        R = _f32(R).reshape(9)
        tc = _f32(tcubes).reshape(-1, 4)
        n = len(tc)
        mask, resid = np.zeros((n, self.Nd), np.uint8), np.zeros((n, self.Nd), np.float32)
        self.eng.check(self.L.goicp_eval_inclusion(self.h, _p(R, C.c_float), int(level), _p(tc, C.c_float), n, mask.ctypes.data_as(C.POINTER(C.c_uint8)), _p(resid, C.c_float)))
        return mask, resid

    def InnerBnB(self, R, level, opt_error):
        """GoICP::InnerBnB (jly_goicp.cpp:286) for n calls: R (n,9), level (n,), opt_error (n,) -> err, tnode, (pops, subcubes)"""
        R = _f32(R).reshape(-1, 9)
        n = len(R)
        level, oe = _i32(np.broadcast_to(level, n)), _f32(np.broadcast_to(opt_error, n))
        err, tn, ps = np.zeros(n, np.float32), np.zeros((n, 4), np.float32), np.zeros((n, 2), np.int64)
        self.eng.check(self.L.goicp_inner_bnb(self.h, _p(R, C.c_float), _p(level, C.c_int32), _p(oe, C.c_float), n, _p(err, C.c_float), _p(tn, C.c_float),
                                              ps.ctypes.data_as(C.POINTER(C.c_int64))))
        return err, tn, ps

    def ICP(self, R, t):
        """GoICP::ICP (jly_goicp.cpp:102)"""
        R, t = _f64(R).reshape(9).copy(), _f64(t).reshape(3).copy()
        err, corr = C.c_float(), np.zeros(self.Nd, np.int32)
        self.eng.check(self.L.goicp_icp(self.h, _p(R, C.c_double), _p(t, C.c_double), C.byref(err), _p(corr, C.c_int32)))
        return float(err.value), R.reshape(3, 3), t, corr

    def Register(self):
        """GoICP::Register (jly_goicp.cpp:878); returns the result dict, also sets optError/optR/optT/optComp."""
        r = Result()
        self.eng.check(self.L.goicp_register(self.h, C.byref(r)))
        d = _result_dict(r)
        d["trace"] = self.L.goicp_last_trace(self.h).decode()
        self.optError, self.optR, self.optT, self.optComp = d["optError"], d["R"], d["t"], d["optComp"]
        return d


def error_trace(trace):
    """The 'Error*:' improvement values of a stdout-style trace."""
    return [line.split()[1].rstrip(",") for line in trace.splitlines() if line.startswith("Error*:")]
