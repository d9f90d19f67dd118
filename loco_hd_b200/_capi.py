"""ctypes binding of the C ABI (include/locohd_b200.h) — used by the parity tests and bench.py so that they call
exactly what a foreign host binding would call.  The Python drop-in API (loco_hd_b200._host, a C++ module) links
the same library directly.

Array arguments may be numpy arrays (host) or integers (raw device pointers, e.g. ``tensor.data_ptr()``).
"""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path
from typing import Optional, Sequence, Tuple

import numpy as np

_PKG = Path(__file__).resolve().parent
LIB_PATH = Path(os.environ["LOCOHD_LIB"]) if os.environ.get("LOCOHD_LIB") else _PKG / "liblocohd_b200.so"   # LOCOHD_LIB: A/B builds

MAX_WF_PARAMS = 16
UNKNOWN_CATEGORY = 0xFFFF
WF_KINDS = {"hyper_exp": 0, "dagum": 1, "uniform": 2, "kumaraswamy": 3}
SD_KINDS = {"Hellinger": 0, "Kolmogorov-Smirnov": 1, "Kullback-Leibler": 2, "Renyi": 3}

# every symbol include/locohd_b200.h declares
EXPORTED_SYMBOLS = [
    "locohd_abi_version", "locohd_device_count", "locohd_ctx_create", "locohd_ctx_destroy", "locohd_last_error",
    "locohd_ctx_set_params", "locohd_ctx_stream", "locohd_ctx_synchronize", "locohd_ctx_launch_count", "locohd_ctx_tile_launches",
    "locohd_ctx_profile_enable", "locohd_ctx_profile_read", "locohd_measure_fp64_tflops",
    "locohd_host_alloc", "locohd_host_free", "locohd_structs_create", "locohd_structs_create_f32",
    "locohd_structs_destroy", "locohd_structs_update_xyz", "locohd_structs_update_xyz_f32",
    "locohd_structs_update_from_atoms", "locohd_structs_drop_cells", "locohd_envset_build", "locohd_envset_from_rows",
    "locohd_envset_from_ragged_rows",
    "locohd_envset_from_coords", "locohd_envset_destroy", "locohd_envset_size", "locohd_envset_total_members",
    "locohd_envset_dump", "locohd_score_pairs", "locohd_score_jobs", "locohd_score_jobs_stats",
    "locohd_score_anchor_lists", "locohd_plan_job_tiles", "locohd_tile_unit", "locohd_tile_geometry",
    "locohd_from_primitives", "locohd_from_primitives_grad", "locohd_from_rows_grad", "locohd_from_coords_grad",
    "locohd_wf_integral_points", "locohd_wf_density_points", "locohd_sd_run",
]


class WeightFunctionC(C.Structure):
    _fields_ = [("kind", C.c_int32), ("n_params", C.c_int32), ("params", C.c_double * MAX_WF_PARAMS)]


class ParamsC(C.Structure):
    _fields_ = [
        ("n_categories", C.c_int32),
        ("category_weights", C.POINTER(C.c_double)),
        ("sd_kind", C.c_int32),
        ("sd_params", C.c_double * 2),
        ("n_weight_functions", C.c_int32),
        ("weight_functions", C.POINTER(WeightFunctionC)),
        ("tpr_kind", C.c_int32),
        ("tpr_accept_same", C.c_int32),
        ("tpr_accepted_pairs", C.c_int32),
        ("tpr_ordered", C.c_int32),
        ("n_tag_pairs", C.c_uint64),
        ("tag_pairs", C.POINTER(C.c_uint64)),
    ]


class JobC(C.Structure):
    _fields_ = [("a_first", C.c_uint64), ("b_first", C.c_uint64), ("n", C.c_uint64)]


JOB_DTYPE = np.dtype([("a_first", "<u8"), ("b_first", "<u8"), ("n", "<u8")])


class LocoHDError(ValueError):
    """Raised for every non-zero status; mirrors the reference's PyValueError (locohd.rs:70-77 etc.)."""

    def __init__(self, status: int, message: str):
        super().__init__(f"[locohd status {status}] {message}")
        self.status = status


_lib = None


def load_library() -> C.CDLL:
    """Load liblocohd_b200.so.  Fails loudly when it has not been built: there is no fallback path."""
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `python loco_hd_b200/build.py` (nvcc, sm_100a). "
            "loco_hd_b200 has no CPU fallback.")
    lib = C.CDLL(str(LIB_PATH))
    vp, u64, i32, u32, dbl = C.c_void_p, C.c_uint64, C.c_int32, C.c_uint32, C.c_double
    sig = {
        "locohd_abi_version": (C.c_int, []),
        "locohd_device_count": (C.c_int, []),
        "locohd_ctx_create": (C.c_int, [C.c_int, C.POINTER(vp)]),
        "locohd_ctx_destroy": (None, [vp]),
        "locohd_last_error": (C.c_char_p, [vp]),
        "locohd_ctx_set_params": (C.c_int, [vp, C.POINTER(ParamsC)]),
        "locohd_ctx_stream": (vp, [vp]),
        "locohd_ctx_synchronize": (C.c_int, [vp]),
        "locohd_ctx_launch_count": (u64, [vp]),
        "locohd_ctx_tile_launches": (u64, [vp]),
        "locohd_ctx_profile_enable": (C.c_int, [vp, C.c_int]),
        "locohd_ctx_profile_read": (C.c_int, [vp, vp, vp]),
        "locohd_measure_fp64_tflops": (C.c_int, [vp, C.POINTER(dbl)]),
        "locohd_host_alloc": (C.c_int, [u64, C.POINTER(vp)]),
        "locohd_host_free": (None, [vp]),
        "locohd_structs_create": (C.c_int, [vp, u64, vp, vp, vp, vp, C.POINTER(vp)]),
        "locohd_structs_create_f32": (C.c_int, [vp, u64, vp, vp, vp, vp, C.POINTER(vp)]),
        "locohd_structs_destroy": (None, [vp]),
        "locohd_structs_update_xyz": (C.c_int, [vp, vp]),
        "locohd_structs_update_xyz_f32": (C.c_int, [vp, vp]),
        "locohd_structs_update_from_atoms": (C.c_int, [vp, u64, u64, u64, vp, u64, vp, vp, u64]),
        "locohd_structs_drop_cells": (None, [vp]),
        "locohd_envset_build": (C.c_int, [vp, vp, u64, vp, vp, dbl, C.c_int, C.POINTER(vp)]),
        "locohd_envset_from_rows": (C.c_int, [vp, u64, u64, vp, vp, C.POINTER(vp)]),
        "locohd_envset_from_ragged_rows": (C.c_int, [vp, u64, vp, vp, vp, u64, C.POINTER(vp)]),
        "locohd_envset_from_coords": (C.c_int, [vp, u64, vp, vp, C.POINTER(vp)]),
        "locohd_envset_destroy": (None, [vp]),
        "locohd_envset_size": (u64, [vp]),
        "locohd_envset_total_members": (u64, [vp]),
        "locohd_envset_dump": (C.c_int, [vp, vp, vp, vp, vp, vp]),
        "locohd_score_pairs": (C.c_int, [vp, vp, vp, u64, vp, vp, vp]),
        "locohd_score_jobs": (C.c_int, [vp, vp, vp, u64, vp, vp, vp, vp]),
        "locohd_score_jobs_stats": (C.c_int, [vp, vp, vp, u64, vp, vp, vp, vp, vp, vp]),
        "locohd_score_anchor_lists": (C.c_int, [vp, vp, u64, vp, u64, vp, u64, vp, u64, u32, vp]),
        "locohd_plan_job_tiles": (C.c_int, [u64, vp, vp, vp, vp]),
        "locohd_tile_unit": (C.c_int, [u64, u64, u64, u64, C.POINTER(u64), C.POINTER(u64)]),
        "locohd_tile_geometry": (C.c_int, [C.c_int, u32, u32, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int),
                                           C.POINTER(C.c_int)]),
        "locohd_from_primitives": (C.c_int, [vp, u64, vp, vp, vp, u64, vp, vp, vp, u64, vp, vp, dbl, vp]),
        "locohd_from_primitives_grad": (C.c_int, [vp, u64, vp, vp, vp, u64, vp, vp, vp, u64, vp, vp, dbl, vp, vp, vp,
                                                  vp]),
        "locohd_from_rows_grad": (C.c_int, [vp, u64, vp, vp, vp, u64, vp, vp, vp, u64, vp, vp, vp, vp, vp]),
        "locohd_from_coords_grad": (C.c_int, [vp, u64, vp, vp, vp, vp, vp, vp, vp, vp, vp]),
        "locohd_wf_integral_points": (C.c_int, [vp, C.POINTER(WeightFunctionC), u64, vp, vp]),
        "locohd_wf_density_points": (C.c_int, [vp, C.POINTER(WeightFunctionC), u64, vp, vp]),
        "locohd_sd_run": (C.c_int, [vp, i32, vp, i32, u64, vp, vp, vp]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def _p(a):
    """numpy array -> host pointer; int -> raw (device) pointer; None -> NULL."""
    if a is None:
        return None
    if isinstance(a, (int, np.integer)):
        return C.c_void_p(int(a))
    return C.c_void_p(a.ctypes.data)


def _arr(a, dtype):
    if a is None or isinstance(a, (int, np.integer)):
        return a
    return np.ascontiguousarray(a, dtype=dtype)


def plan_job_tiles(jobs) -> dict:
    """locohd_plan_job_tiles: how a job list groups into tiles of jobs that share runs of environments (host-side
    query, no device needed).  Returns {"tiles", "rows", "pays"}."""
    lib = load_library()
    jobs = np.ascontiguousarray(jobs, dtype=JOB_DTYPE)
    tiles, rows, pays = C.c_uint64(0), C.c_uint64(0), C.c_int(0)
    st = lib.locohd_plan_job_tiles(len(jobs), _p(jobs), C.byref(tiles), C.byref(rows), C.byref(pays))
    if st:
        raise LocoHDError(st, "locohd_plan_job_tiles failed")
    return {"tiles": int(tiles.value), "rows": int(rows.value), "pays": bool(pays.value)}


def tile_unit(n_tiles: int, n_anchors: int, slice_: int, unit: int):
    """(tile, anchor) at position `unit` of a tile launch (locohd_tile_unit; host-side, no device)."""
    t, p = C.c_uint64(), C.c_uint64()
    st = load_library().locohd_tile_unit(n_tiles, n_anchors, slice_, unit, C.byref(t), C.byref(p))
    if st:
        raise LocoHDError(st, "locohd_tile_unit")
    return int(t.value), int(p.value)


def tile_geometry(n_categories: int, max_a: int, max_b: int) -> dict:
    """Launch geometry of the tile kernel for environments of at most max_a / max_b members (locohd_tile_geometry;
    host-side, no device).  Returns {"teams", "cp", "rep_n", "table_n"}; teams == 0: the tile kernel does not apply,
    and jobs take it only from 6 teams on."""
    teams, cp, rep_n, table_n = C.c_int(), C.c_int(), C.c_int(), C.c_int()
    st = load_library().locohd_tile_geometry(n_categories, max_a, max_b, C.byref(teams), C.byref(cp), C.byref(rep_n),
                                             C.byref(table_n))
    if st:
        raise LocoHDError(st, "locohd_tile_geometry")
    return {"teams": teams.value, "cp": cp.value, "rep_n": rep_n.value, "table_n": table_n.value}


def make_wf(name: str, params: Sequence[float]) -> WeightFunctionC:
    w = WeightFunctionC()
    w.kind = WF_KINDS[name]
    params = list(params)
    if len(params) > MAX_WF_PARAMS:
        raise LocoHDError(10, f"at most {MAX_WF_PARAMS} weight function parameters are supported")
    w.n_params = len(params)
    for i, v in enumerate(params):
        w.params[i] = float(v)
    return w


class Context:
    """One GPU context (locohd_ctx)."""

    def __init__(self, device: int = 0):
        self.lib = load_library()
        h = C.c_void_p()
        st = self.lib.locohd_ctx_create(device, C.byref(h))
        if st:
            raise LocoHDError(st, self.lib.locohd_last_error(None).decode())
        self.h = h
        self.device = device
        self.n_categories = 0

    def close(self):
        if getattr(self, "h", None):
            self.lib.locohd_ctx_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, st: int):
        if st:
            raise LocoHDError(st, self.lib.locohd_last_error(self.h).decode())

    @property
    def stream(self) -> int:
        return int(self.lib.locohd_ctx_stream(self.h) or 0)

    @property
    def launch_count(self) -> int:
        return int(self.lib.locohd_ctx_launch_count(self.h))

    @property
    def tile_launches(self) -> int:
        return int(self.lib.locohd_ctx_tile_launches(self.h))

    def synchronize(self):
        self._check(self.lib.locohd_ctx_synchronize(self.h))

    PROF_GROUPS = ("cells", "count", "scan", "fill", "score", "other", "sort")

    def profile_enable(self, on: bool = True):
        self._check(self.lib.locohd_ctx_profile_enable(self.h, int(on)))

    def profile_read(self):
        """-> {group: (total ms, launch groups)} accumulated since the last read."""
        ms = np.zeros(len(self.PROF_GROUPS), np.float64)
        n = np.zeros(len(self.PROF_GROUPS), np.uint64)
        self._check(self.lib.locohd_ctx_profile_read(self.h, _p(ms), _p(n)))
        return {g: (float(ms[i]), int(n[i])) for i, g in enumerate(self.PROF_GROUPS)}

    def measure_fp64_tflops(self) -> float:
        out = C.c_double()
        self._check(self.lib.locohd_measure_fp64_tflops(self.h, C.byref(out)))
        return out.value

    def host_alloc(self, nbytes: int) -> int:
        h = C.c_void_p()
        st = self.lib.locohd_host_alloc(int(nbytes), C.byref(h))
        if st:
            raise LocoHDError(st, self.lib.locohd_last_error(None).decode())
        return int(h.value)

    def host_free(self, ptr: int):
        self.lib.locohd_host_free(C.c_void_p(ptr))

    def pinned_array(self, shape, dtype):
        """numpy array backed by pinned host memory (kept alive by the returned array's base object)."""
        dtype = np.dtype(dtype)
        n = int(np.prod(shape)) * dtype.itemsize
        ptr = self.host_alloc(max(n, 1))
        buf = (C.c_char * max(n, 1)).from_address(ptr)
        arr = np.frombuffer(buf, dtype=dtype, count=int(np.prod(shape))).reshape(shape)
        self._pinned = getattr(self, "_pinned", [])
        self._pinned.append(ptr)
        return arr

    def set_params(self, n_categories: int, weight_functions=(("uniform", (3.0, 10.0)),), category_weights=None,
                   statistical_distance=("Hellinger", (2.0,)), tag_rule=None):
        """tag_rule: {"accept_same": bool} or {"tag_pairs": [(a, b), ...], "accepted_pairs": bool, "ordered": bool}
        on interned tag ids; None = the reference's default accept_same=True (locohd.rs:357-362)."""
        p = ParamsC()
        p.n_categories = n_categories
        cw = None
        if category_weights is not None:
            cw = np.ascontiguousarray(category_weights, dtype=np.float64)
            if len(cw) != n_categories:
                raise LocoHDError(10, "LoCoHD parameters 'categories' and 'category_weights' must have the same lengths!")
            p.category_weights = cw.ctypes.data_as(C.POINTER(C.c_double))
        name, sdp = statistical_distance
        p.sd_kind = SD_KINDS[name]
        sdp = list(sdp) + [0.0, 0.0]
        p.sd_params[0], p.sd_params[1] = float(sdp[0]), float(sdp[1])
        wfs = (WeightFunctionC * len(weight_functions))(*[make_wf(n, q) for n, q in weight_functions])
        p.n_weight_functions = len(weight_functions)
        p.weight_functions = wfs
        rule = {"accept_same": True} if tag_rule is None else tag_rule
        pairs = None
        if "accept_same" in rule:
            p.tpr_kind, p.tpr_accept_same = 0, int(bool(rule["accept_same"]))
        else:
            p.tpr_kind = 1
            p.tpr_accepted_pairs = int(bool(rule["accepted_pairs"]))
            p.tpr_ordered = int(bool(rule["ordered"]))
            pairs = np.array([(int(a) << 32) | int(b) for a, b in rule["tag_pairs"]] or [0], dtype=np.uint64)
            p.n_tag_pairs = len(rule["tag_pairs"])
            p.tag_pairs = pairs.ctypes.data_as(C.POINTER(C.c_uint64))
        self._check(self.lib.locohd_ctx_set_params(self.h, C.byref(p)))
        self.n_categories = n_categories

    # ---- structures -------------------------------------------------------------------------------
    def structs_create(self, prim_offsets, xyz, category, tag, f32: Optional[bool] = None) -> "Structs":
        """xyz: float64 array (or raw pointer) -> locohd_structs_create; float32 array (or raw pointer with
        f32=True) -> locohd_structs_create_f32 (half the upload, widened exactly on the device)."""
        offs = np.ascontiguousarray(prim_offsets, dtype=np.uint64)
        if f32 is None:
            f32 = isinstance(xyz, np.ndarray) and xyz.dtype == np.float32
        xyz = _arr(xyz, np.float32 if f32 else np.float64)
        category, tag = _arr(category, np.uint16), _arr(tag, np.uint32)
        h = C.c_void_p()
        fn = self.lib.locohd_structs_create_f32 if f32 else self.lib.locohd_structs_create
        self._check(fn(self.h, len(offs) - 1, _p(offs), _p(xyz), _p(category), _p(tag), C.byref(h)))
        return Structs(self, h, len(offs) - 1, int(offs[-1]))

    def structure(self, xyz, category, tag) -> "Structs":
        n = len(category)
        return self.structs_create([0, n], xyz, category, tag)

    # ---- environments -----------------------------------------------------------------------------
    def envset_build(self, structs: "Structs", anchor_prim, threshold: float, anchor_struct=None,
                     keep_indices: bool = False, n_anchors: Optional[int] = None) -> "EnvSet":
        ap, as_ = _arr(anchor_prim, np.uint32), _arr(anchor_struct, np.uint32)
        n = int(n_anchors) if n_anchors is not None else len(ap)
        h = C.c_void_p()
        self._check(self.lib.locohd_envset_build(self.h, structs.h, n, _p(as_), _p(ap), float(threshold),
                                                 int(keep_indices), C.byref(h)))
        return EnvSet(self, h)

    def envset_from_rows(self, dmx, category) -> "EnvSet":
        dmx = np.ascontiguousarray(dmx, dtype=np.float64)
        dmx = dmx.reshape(len(dmx), -1)
        cat = np.ascontiguousarray(category, dtype=np.uint16)
        h = C.c_void_p()
        self._check(self.lib.locohd_envset_from_rows(self.h, dmx.shape[0], dmx.shape[1], _p(dmx), _p(cat), C.byref(h)))
        return EnvSet(self, h)

    def envset_from_ragged_rows(self, rows, category) -> "EnvSet":
        """rows: sequence of 1-D distance arrays of different lengths (locohd_envset_from_ragged_rows)."""
        rows = [np.ascontiguousarray(r, dtype=np.float64).ravel() for r in rows]
        offs = np.cumsum([0] + [len(r) for r in rows]).astype(np.uint64)
        vals = np.concatenate(rows) if rows else np.zeros(0)
        cat = np.ascontiguousarray(category, dtype=np.uint16)
        h = C.c_void_p()
        self._check(self.lib.locohd_envset_from_ragged_rows(self.h, len(rows), _p(offs), _p(vals), _p(cat), len(cat),
                                                            C.byref(h)))
        return EnvSet(self, h)

    def envset_from_coords(self, xyz, category) -> "EnvSet":
        xyz = np.ascontiguousarray(xyz, dtype=np.float64).reshape(-1, 3)
        cat = np.ascontiguousarray(category, dtype=np.uint16)
        h = C.c_void_p()
        self._check(self.lib.locohd_envset_from_coords(self.h, len(xyz), _p(xyz), _p(cat), C.byref(h)))
        return EnvSet(self, h)

    # ---- scoring ----------------------------------------------------------------------------------
    def score_pairs(self, a: "EnvSet", b: "EnvSet", pairs, wf_idx=None, out=None, n_pairs: Optional[int] = None):
        pairs, wf_idx = _arr(pairs, np.uint32), _arr(wf_idx, np.uint32)
        n = int(n_pairs) if n_pairs is not None else len(pairs.reshape(-1, 2))
        res = np.empty(n, np.float64) if out is None else out
        self._check(self.lib.locohd_score_pairs(self.h, a.h, b.h, n, _p(pairs), _p(wf_idx), _p(res)))
        return res

    def score_jobs_stats(self, a: "EnvSet", b: "EnvSet", jobs, wf_idx=None, scores=False, job_means=False,
                         anchor_means=False, anchor_stds=False):
        """locohd_score_jobs_stats: returns a dict with the requested arrays (each flag may also be an output array
        or a raw device pointer).  The per-anchor statistics need jobs of one common size."""
        jobs = np.ascontiguousarray(jobs, dtype=JOB_DTYPE)
        wf_idx = _arr(wf_idx, np.uint32)
        total = int(jobs["n"].sum())
        n = int(jobs["n"][0]) if len(jobs) else 0

        def buf(flag, size):
            if flag is False or flag is None:
                return None
            return np.empty(size, np.float64) if flag is True else flag

        res = {"scores": buf(scores, total), "job_means": buf(job_means, len(jobs)),
               "anchor_means": buf(anchor_means, n), "anchor_stds": buf(anchor_stds, n)}
        self._check(self.lib.locohd_score_jobs_stats(self.h, a.h, b.h, len(jobs), _p(jobs), _p(wf_idx),
                                                     _p(res["scores"]), _p(res["job_means"]), _p(res["anchor_means"]),
                                                     _p(res["anchor_stds"])))
        return {k: v for k, v in res.items() if v is not None}

    def score_jobs(self, a: "EnvSet", b: "EnvSet", jobs, wf_idx=None, out=None, want_scores=True, want_means=False,
                   means_out=None):
        """`out` / `means_out`: numpy array (host) or raw device pointer; with `want_scores=False` and a `means_out`
        only the per-job means leave the device (SURVEY 8(f) N4: the 1000-structure ensemble would otherwise copy
        20 GB of per-anchor scores back)."""
        jobs = np.ascontiguousarray(jobs, dtype=JOB_DTYPE) if not isinstance(jobs, np.ndarray) or jobs.dtype != JOB_DTYPE \
            else np.ascontiguousarray(jobs)
        wf_idx = _arr(wf_idx, np.uint32)
        total = int(jobs["n"].sum())
        res = out if out is not None else (np.empty(total, np.float64) if want_scores else None)
        want_means = want_means or means_out is not None
        means = means_out if means_out is not None else (np.empty(len(jobs), np.float64) if want_means else None)
        self._check(self.lib.locohd_score_jobs(self.h, a.h, b.h, len(jobs), _p(jobs), _p(wf_idx), _p(res), _p(means)))
        if want_means:
            return res, means
        return res

    def score_anchor_lists(self, seq_a, dists_a, seq_b, dists_b, wf_idx: int = 0) -> float:
        sa, sb = np.ascontiguousarray(seq_a, dtype=np.uint16), np.ascontiguousarray(seq_b, dtype=np.uint16)
        da, db = np.ascontiguousarray(dists_a, dtype=np.float64), np.ascontiguousarray(dists_b, dtype=np.float64)
        out = np.zeros(1, np.float64)
        self._check(self.lib.locohd_score_anchor_lists(self.h, _p(sa), len(sa), _p(da), len(da), _p(sb), len(sb),
                                                       _p(db), len(db), wf_idx, _p(out)))
        return float(out[0])

    def from_primitives(self, xyz_a, cat_a, tag_a, xyz_b, cat_b, tag_b, anchors, threshold: float, wf_idx=None,
                        out=None, n_a=None, n_b=None, n_pairs=None):
        xyz_a, xyz_b = _arr(xyz_a, np.float64), _arr(xyz_b, np.float64)
        cat_a, cat_b = _arr(cat_a, np.uint16), _arr(cat_b, np.uint16)
        tag_a, tag_b = _arr(tag_a, np.uint32), _arr(tag_b, np.uint32)
        anchors, wf_idx = _arr(anchors, np.uint32), _arr(wf_idx, np.uint32)
        na = int(n_a) if n_a is not None else len(cat_a)
        nb = int(n_b) if n_b is not None else len(cat_b)
        P = int(n_pairs) if n_pairs is not None else len(anchors.reshape(-1, 2))
        res = np.empty(P, np.float64) if out is None else out
        self._check(self.lib.locohd_from_primitives(self.h, na, _p(xyz_a), _p(cat_a), _p(tag_a), nb, _p(xyz_b),
                                                    _p(cat_b), _p(tag_b), P, _p(anchors), _p(wf_idx),
                                                    float(threshold), _p(res)))
        return res

    def from_primitives_grad(self, xyz_a, cat_a, tag_a, xyz_b, cat_b, tag_b, anchors, threshold: float, wf_idx=None,
                             pair_weights=None, out=None, grad_a=None, grad_b=None, n_a=None, n_b=None, n_pairs=None):
        """Scores and their coordinate gradients: returns (scores [P], grad_a [n_a, 3], grad_b [n_b, 3]) with
        grad = sum_p pair_weights[p] dS_p/dxyz (pair_weights None: all 1).  Every array may be a numpy array or a raw
        device pointer, as in from_primitives."""
        xyz_a, xyz_b = _arr(xyz_a, np.float64), _arr(xyz_b, np.float64)
        cat_a, cat_b = _arr(cat_a, np.uint16), _arr(cat_b, np.uint16)
        tag_a, tag_b = _arr(tag_a, np.uint32), _arr(tag_b, np.uint32)
        anchors, wf_idx = _arr(anchors, np.uint32), _arr(wf_idx, np.uint32)
        pair_weights = _arr(pair_weights, np.float64)
        na = int(n_a) if n_a is not None else len(cat_a)
        nb = int(n_b) if n_b is not None else len(cat_b)
        P = int(n_pairs) if n_pairs is not None else len(anchors.reshape(-1, 2))
        res = np.empty(P, np.float64) if out is None else out
        ga = np.empty((na, 3), np.float64) if grad_a is None else grad_a
        gb = np.empty((nb, 3), np.float64) if grad_b is None else grad_b
        self._check(self.lib.locohd_from_primitives_grad(self.h, na, _p(xyz_a), _p(cat_a), _p(tag_a), nb, _p(xyz_b),
                                                         _p(cat_b), _p(tag_b), P, _p(anchors), _p(wf_idx),
                                                         float(threshold), _p(pair_weights), _p(res), _p(ga), _p(gb)))
        return res, ga, gb

    def from_rows_grad(self, rows_a, cat_a, rows_b, cat_b, wf_idx=None, pair_weights=None, out=None, grad_a=None,
                       grad_b=None, offsets_a=None, offsets_b=None, n_rows=None):
        """from_dmxs scores with the gradient of row r's score with respect to every entry of row r of either side:
        returns (scores [n_rows], grad_a, grad_b), grad = pair_weights[r] dS_r / d entry (pair_weights None: all 1).
        rows_s is a 2-D array (grads come back [n_rows, row_len]) or a list of 1-D rows (grads come back as a list of
        1-D arrays).  With offsets_s given, rows_s is the flat values (numpy or a raw device pointer) of ragged rows
        at those offsets and grad_s comes back flat in the same layout.  wf_idx, pair_weights, out, grad_a and grad_b
        may be raw device pointers."""
        def flat(rows, offsets):
            if offsets is not None:
                offsets = _arr(offsets, np.uint64)
                return _arr(rows, np.float64), offsets, lambda g: g
            if not isinstance(rows, np.ndarray):
                try:
                    rows = np.asarray(rows, dtype=np.float64)
                except ValueError:   # ragged
                    rows = [np.ascontiguousarray(r, dtype=np.float64).ravel() for r in rows]
                    offs = np.cumsum([0] + [len(r) for r in rows]).astype(np.uint64)
                    vals = np.concatenate(rows) if rows else np.zeros(0)
                    return vals, offs, lambda g: np.split(g, offs[1:-1]) if len(rows) else []
            rows = np.ascontiguousarray(rows, dtype=np.float64)
            if rows.ndim != 2:
                rows = rows.reshape(len(rows), -1)
            offs = (np.arange(rows.shape[0] + 1) * rows.shape[1]).astype(np.uint64)
            return rows.ravel(), offs, lambda g: g.reshape(rows.shape)

        va, oa, shape_a = flat(rows_a, offsets_a)
        vb, ob, shape_b = flat(rows_b, offsets_b)
        n = int(n_rows) if n_rows is not None else len(oa) - 1
        cat_a, cat_b = _arr(cat_a, np.uint16), _arr(cat_b, np.uint16)
        wf_idx, pair_weights = _arr(wf_idx, np.uint32), _arr(pair_weights, np.float64)
        res = np.empty(n, np.float64) if out is None else out
        ga = np.empty(int(oa[n]), np.float64) if grad_a is None else grad_a
        gb = np.empty(int(ob[n]), np.float64) if grad_b is None else grad_b
        self._check(self.lib.locohd_from_rows_grad(self.h, n, _p(oa), _p(va), _p(cat_a), len(cat_a), _p(ob), _p(vb),
                                                   _p(cat_b), len(cat_b), _p(wf_idx), _p(pair_weights), _p(res),
                                                   _p(ga), _p(gb)))
        return (res, shape_a(ga) if grad_a is None else ga, shape_b(gb) if grad_b is None else gb)

    def from_coords_grad(self, xyz_a, cat_a, xyz_b, cat_b, wf_idx=None, pair_weights=None, out=None, grad_a=None,
                         grad_b=None, n_points=None):
        """from_coords scores and their coordinate gradients: (scores [n], grad_a [n, 3], grad_b [n, 3]) with
        grad = sum_r pair_weights[r] dS_r/dxyz (pair_weights None: all 1).  Every array may be a numpy array or a
        raw device pointer (then n_points is needed)."""
        xyz_a, xyz_b = _arr(xyz_a, np.float64), _arr(xyz_b, np.float64)
        cat_a, cat_b = _arr(cat_a, np.uint16), _arr(cat_b, np.uint16)
        wf_idx, pair_weights = _arr(wf_idx, np.uint32), _arr(pair_weights, np.float64)
        n = int(n_points) if n_points is not None else len(xyz_a.reshape(-1, 3))
        res = np.empty(n, np.float64) if out is None else out
        ga = np.empty((n, 3), np.float64) if grad_a is None else grad_a
        gb = np.empty((n, 3), np.float64) if grad_b is None else grad_b
        self._check(self.lib.locohd_from_coords_grad(self.h, n, _p(xyz_a), _p(cat_a), _p(xyz_b), _p(cat_b),
                                                     _p(wf_idx), _p(pair_weights), _p(res), _p(ga), _p(gb)))
        return res, ga, gb

    # ---- leaf math --------------------------------------------------------------------------------
    def wf_integral_points(self, name: str, params, x):
        w = make_wf(name, params)
        x = np.ascontiguousarray(x, dtype=np.float64)
        out = np.empty(len(x), np.float64)
        self._check(self.lib.locohd_wf_integral_points(self.h, C.byref(w), len(x), _p(x), _p(out)))
        return out

    def wf_density_points(self, name: str, params, x):
        """The weight function's density dW/dx at the points x."""
        w = make_wf(name, params)
        x = np.ascontiguousarray(x, dtype=np.float64)
        out = np.empty(len(x), np.float64)
        self._check(self.lib.locohd_wf_density_points(self.h, C.byref(w), len(x), _p(x), _p(out)))
        return out

    def sd_run(self, name: str, params, p1, p2):
        p1 = np.ascontiguousarray(p1, dtype=np.float64)
        p2 = np.ascontiguousarray(p2, dtype=np.float64)
        p1 = p1.reshape(-1, p1.shape[-1])
        p2 = p2.reshape(-1, p2.shape[-1])
        sdp = np.asarray(list(params) + [0.0, 0.0], dtype=np.float64)
        out = np.empty(len(p1), np.float64)
        self._check(self.lib.locohd_sd_run(self.h, SD_KINDS[name], _p(sdp), p1.shape[1], len(p1), _p(p1), _p(p2),
                                           _p(out)))
        return out


class Structs:
    def __init__(self, ctx: Context, h, n_structs: int, n_prims: int):
        self.ctx, self.h, self.n_structs, self.n_prims = ctx, h, n_structs, n_prims

    def update_xyz(self, xyz, f32: Optional[bool] = None):
        if f32 is None:
            f32 = isinstance(xyz, np.ndarray) and xyz.dtype == np.float32
        if f32:
            self.ctx._check(self.ctx.lib.locohd_structs_update_xyz_f32(self.h, _p(_arr(xyz, np.float32))))
        else:
            self.ctx._check(self.ctx.lib.locohd_structs_update_xyz(self.h, _p(_arr(xyz, np.float64))))

    def update_from_atoms(self, atom_xyz, segment_start, atom_index, first_struct: int = 0, n_frames: int = 1,
                          n_atoms: Optional[int] = None):
        """Frames of one compiled topology (PrimitiveAssigner.compile_topology): atom_xyz [n_frames][n_atoms][3]
        float32 -> primitive centroids of structures [first_struct, first_struct + n_frames) on the device."""
        seg, idx = _arr(segment_start, np.uint32), _arr(atom_index, np.uint32)
        atoms = _arr(atom_xyz, np.float32)
        if n_atoms is None:
            n_atoms = atoms.size // (3 * n_frames)
        self.ctx._check(self.ctx.lib.locohd_structs_update_from_atoms(
            self.h, int(first_struct), int(n_frames), int(n_atoms), _p(atoms), len(seg) - 1, _p(seg), _p(idx), len(idx)))

    def drop_cells(self):
        self.ctx.lib.locohd_structs_drop_cells(self.h)

    def close(self):
        if self.h and self.ctx.h:
            self.ctx.lib.locohd_structs_destroy(self.h)
        self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class EnvSet:
    def __init__(self, ctx: Context, h):
        self.ctx, self.h = ctx, h

    def __len__(self):
        return int(self.ctx.lib.locohd_envset_size(self.h))

    @property
    def total_members(self) -> int:
        return int(self.ctx.lib.locohd_envset_total_members(self.h))

    def dump(self, indices: bool = True):
        """-> offsets [n+1], distances, categories, primitive indices (or None)."""
        n, tot = len(self), self.total_members
        off = np.empty(n + 1, np.uint64)
        d = np.empty(tot, np.float64)
        c = np.empty(tot, np.uint16)
        ix = np.empty(tot, np.uint32) if indices else None
        self.ctx._check(self.ctx.lib.locohd_envset_dump(self.ctx.h, self.h, _p(off), _p(d), _p(c), _p(ix)))
        return off, d, c, ix

    def close(self):
        if self.h and self.ctx.h:
            self.ctx.lib.locohd_envset_destroy(self.h)
        self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
