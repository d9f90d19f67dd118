#!/usr/bin/env python
"""bench.py — LoCoHD anchor-pairs/second on B200 (BASELINE.json metric), one process per GPU.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload cfg5|cfg2|cfg3|cfg4] [--impl reference]

A *step* is one pass of the hot path over one batch of synthetic structures (SURVEY.md §8(d) generator):
cell lists (K0) -> environments (K1) -> scoring (K2) -> reductions.

Default workload = the north-star target of BASELINE.json (configs[4]): the all-vs-all ensemble of 1000 structures x
5000 primitives (all_atom shape, C = 7), uniform [3, 10], 10 A threshold, hetero contacts only, every primitive an
anchor: 499 500 structure pairs = 2.4975e9 anchor pairs per step, dealt round-robin over the GPUs (strong scaling: the
whole ensemble is resident on every GPU, no collective on the scoring path).  Only the per-structure-pair means leave
the device (what compare_ensembles.py:293 computes from the scores; 20 GB of per-anchor scores stay in device scratch).
At N = 1 the line also carries one short run each of configs[1..3] (`other_workloads`) and the Python-API call
latencies (`e2e_python`).  `--workload cfg2|cfg3|cfg4` makes one of those the main workload (weak scaling).

    value  whole-job throughput with the structures already resident in HBM (CUDA events on the library stream)
    e2e    same metric through the C-ABI call sequence with HOST (pinned) buffers: H2D of the structures and
           anchors and D2H of the results inside the timed region (wall clock between synchronisations); short
           steps are also measured with two host threads / contexts (the copies of one step overlap the kernels of
           the other) and `e2e.value` is the better of the two, both are in the line

`--dump-outputs DIR` writes what the last timed step returned (job_means.npy or scores.npy, float64) for comparing two
builds output for output; the inputs depend only on the arguments (seeded generator).

`--impl reference` times the CPU restatement of the reference algorithm (oracle/, all host threads; the Rust crate
cannot be built in this image) on a bounded sample of the same workload.  That arm imports only `benchdata` and
`oracle`: it never maps the CUDA library.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
if str(ROOT) not in sys.path:
    sys.path.insert(0, str(ROOT))
sys.dont_write_bytecode = True   # the benchmark leaves the tree as it found it (it may be read-only)



def _ensure_built():
    """A clean checkout has no built extension (the .so files are git-ignored): build it through build.py loaded by
    path (the package cannot be imported before).  Rank 0 of a multi-process launch builds, the others wait."""
    import importlib.util
    import sysconfig

    pkg = ROOT / "loco_hd_b200"
    need = [pkg / "liblocohd_b200.so", ROOT / "loco_hd" / ("loco_hd" + sysconfig.get_config_var("EXT_SUFFIX"))]
    if all(p.exists() for p in need):
        return
    if int(os.environ.get("LOCAL_RANK", "0")) == 0:
        spec = importlib.util.spec_from_file_location("_locohd_build", pkg / "build.py")
        b = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(b)
        b.build_all()
    else:
        for _ in range(600):
            if all(p.exists() for p in need):
                break
            time.sleep(1.0)
        time.sleep(2.0)


from benchdata import synth  # noqa: E402  (no product code: the reference arm must not map the CUDA library)


def _load_batch_helpers():
    """loco_hd_b200/batch.py (pure numpy job dealing) loaded by path: importing the package would map the CUDA library,
    which the CPU reference arm must not do."""
    import importlib.util

    spec = importlib.util.spec_from_file_location("_locohd_batch", ROOT / "loco_hd_b200" / "batch.py")
    mod = importlib.util.module_from_spec(spec)
    sys.modules[spec.name] = mod   # dataclasses resolve the module of a class through sys.modules
    spec.loader.exec_module(mod)
    return mod.blocked_pairs, mod.contiguous_share


blocked_pairs, contiguous_share = _load_batch_helpers()

F_WF = {"uniform": 11, "kumaraswamy": 19, "dagum": 9}  # SURVEY.md §8(d): flops of one integral_range


# ------------------------------------------------------------------------------------------------ workloads
class Workload:
    """clouds: structures of this rank; groups: (structure, anchor primitive indices) -> one environment each,
    laid out group after group; jobs: (group_a, group_b) scored with identity pairing."""

    def __init__(self, name, desc, n_categories, wf, clouds, groups, jobs, scaling="weak", means_only=False):
        self.name, self.desc, self.C, self.wf, self.scaling = name, desc, n_categories, wf, scaling
        self.means_only = means_only
        self.rule = {"accept_same": False}
        self.threshold = 10.0
        self.clouds = clouds
        self.offsets = np.cumsum([0] + [c.n for c in clouds]).astype(np.uint64)
        self.xyz = np.concatenate([c.xyz for c in clouds])
        self.cat = np.concatenate([c.cat for c in clouds]).astype(np.uint16)
        self.tag = np.concatenate([c.tag for c in clouds]).astype(np.uint32)
        self.anchor_struct = np.concatenate([np.full(len(p), s, np.uint32) for s, p in groups])
        self.anchor_prim = np.concatenate([np.asarray(p, np.uint32) for _, p in groups])
        goff = np.cumsum([0] + [len(p) for _, p in groups])
        self.jobs = np.empty(len(jobs), dtype=[("a_first", "<u8"), ("b_first", "<u8"), ("n", "<u8")])
        if len(jobs):
            ja = np.asarray(jobs, dtype=np.int64).reshape(-1, 2)
            self.jobs["a_first"], self.jobs["b_first"] = goff[ja[:, 0]], goff[ja[:, 1]]
            self.jobs["n"] = goff[ja[:, 0] + 1] - goff[ja[:, 0]]
        self.n_pairs = int(self.jobs["n"].sum())
        self.groups, self.job_groups = groups, jobs

    @property
    def h2d_bytes(self):
        return (self.xyz.nbytes + self.cat.nbytes + self.tag.nbytes + self.offsets.nbytes + self.anchor_struct.nbytes
                + self.anchor_prim.nbytes + self.jobs.nbytes)

    def job_arrays(self, j):
        """(A cloud, B cloud, anchors [n, 2]) of job j, for the CPU restatement."""
        ga, gb = self.job_groups[j]
        (sa, pa), (sb, pb) = self.groups[ga], self.groups[gb]
        return self.clouds[sa], self.clouds[sb], np.stack([pa, pb], axis=1).astype(np.uint32)


def make_workload(name, rank, world, args):
    if name == "cfg2":
        B = args.pairs
        clouds, groups, jobs = [], [], []
        for i in range(B):
            a, b = synth.config2_pair(rank * B + i)
            clouds += [a, b]
            groups += [(2 * i, np.arange(a.n)), (2 * i + 1, np.arange(b.n))]
            jobs.append((2 * i, 2 * i + 1))
        return Workload("cfg2", f"BASELINE configs[1]: {B} all_atom-shaped structure pairs per GPU (10000 primitives each, "
                        "C=7), kumaraswamy [3,10,2,5], threshold 10, accept_same=False, every primitive an anchor",
                        7, ("kumaraswamy", (3.0, 10.0, 2.0, 5.0)), clouds, groups, jobs)
    if name == "cfg3":
        M = args.models
        ref = synth.config3_reference()
        clouds = [ref] + [synth.config3_model(ref, rank * M + m) for m in range(M)]
        cent = ref.centroid_anchors()
        groups = [(s, cent) for s in range(M + 1)]
        return Workload("cfg3", f"BASELINE configs[2]: 1 reference vs {M} models per GPU (300 residues, 2700 primitives, "
                        "all_atom_with_centroid, C=8), uniform [3,10], Cent anchors", 8, ("uniform", (3.0, 10.0)), clouds,
                        groups, [(0, m + 1) for m in range(M)])
    if name == "cfg4":
        F = args.frames
        f0 = synth.config4_frame0()
        clouds = [f0] + [synth.config4_frame(f0, 1 + rank * F + t) for t in range(F)]
        cent = f0.centroid_anchors()
        groups = [(s, cent) for s in range(F + 1)]
        return Workload("cfg4", f"BASELINE configs[3]: {F} trajectory frames per GPU (5000 primitives, "
                        "coarse_grained_with_centroid, C=8) vs frame 0, uniform [3,10], 1250 Cent anchors per frame", 8,
                        ("uniform", (3.0, 10.0)), clouds, groups, [(0, t + 1) for t in range(F)])
    if name == "cfg5":
        S = args.ensemble
        base = synth.config5_base()
        clouds = [synth.config5_member(base, i) for i in range(S)]
        groups = [(s, np.arange(base.n)) for s in range(S)]
        # all i < j structure pairs, in 4 x 4 tiles of the upper triangle (8 structures' environments = 61 MB stay in
        # L2 while 16 structure pairs are scored); every rank takes one contiguous run of that list
        all_jobs = blocked_pairs(S, int(os.environ.get("LOCOHD_BENCH_BLOCK", "4")))
        mine = all_jobs[contiguous_share(len(all_jobs), rank, world)]
        return Workload("cfg5", f"BASELINE configs[4]: all-vs-all ensemble of {S} structures (5000 primitives, all_atom, "
                        f"C=7), uniform [3,10], every primitive an anchor; {len(all_jobs)} structure pairs in 4x4 tiles, "
                        f"one contiguous run per GPU ({world} GPU(s))", 7, ("uniform", (3.0, 10.0)), clouds, groups,
                        [tuple(q) for q in mine.tolist()], scaling="strong", means_only=True)
    raise SystemExit(f"unknown workload {name}")


# ---------------------------------------------------------------------------------------------------- clocks
class ClockSampler:
    """SM clock / throttle reasons sampled DURING the timed region through NVML (in-process, ~20 Hz).  A looping
    `nvidia-smi -lms` next to the benchmark perturbs short kernels on these hosts, so it is only the fallback."""

    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, device):
        self.rows, self.stop_flag, self.nvml, self.proc = [], False, None, None
        self.period = float(os.environ.get("LOCOHD_BENCH_CLOCK_PERIOD", "0.05"))
        try:
            import pynvml

            pynvml.nvmlInit()
            # NVML enumerates physical devices: map through CUDA_VISIBLE_DEVICES when it is a plain index list
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            idx = device
            if vis and all(v.strip().isdigit() for v in vis.split(",")):
                idx = int(vis.split(",")[device])
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(idx)
            self.nvml = pynvml
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM))
        except Exception:
            self.nvml = None
        self.thread = threading.Thread(target=self._poll if self.nvml else self._smi, args=(device,), daemon=True)
        self.thread.start()

    def _poll(self, device):
        n = self.nvml
        while not self.stop_flag:
            try:
                mhz = float(n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM))
                try:
                    mask = int(n.nvmlDeviceGetCurrentClocksEventReasons(self.handle))
                except Exception:
                    mask = int(n.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle))
                self.rows.append((time.perf_counter(), mhz, self.max_mhz, mask))
            except Exception:
                pass
            time.sleep(self.period)

    def _smi(self, device):
        fields = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
                  "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={fields}", "--format=csv,noheader,nounits", "-i",
                                      str(device)], capture_output=True, text=True, timeout=5).stdout.strip()
                v = [x.strip() for x in out.split(",")]
                mask = sum(bit for bit, flag in zip((0x8, 0x40, 0x20, 0x4), v[2:6]) if flag == "Active")
                self.rows.append((time.perf_counter(), float(v[0]), float(v[1]), mask))
            except Exception:
                pass
            time.sleep(1.0)

    def stop(self, t_begin=None, t_end=None):
        """Summary of the samples taken inside [t_begin, t_end] (the timed region)."""
        self.stop_flag = True
        self.thread.join(timeout=3)
        rows = [r for r in self.rows if (t_begin is None or r[0] >= t_begin) and (t_end is None or r[0] <= t_end)]
        if not rows:
            rows = self.rows[-3:]
        if not rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no clock samples"], "samples": 0}
        mask = 0
        for r in rows:
            mask |= r[3]
        reasons = sorted(name for bit, name in self.REASONS.items() if mask & bit)
        return {"sm_mhz": float(np.median([r[1] for r in rows])), "sm_max_mhz": max(r[2] for r in rows),
                "reasons": reasons, "samples": len(rows), "source": "nvml" if self.nvml else "nvidia-smi"}


# --------------------------------------------------------------------------------------------- reference arm
def oracle_params(oracle, wl):
    return oracle.Params(wl.C, [(wl.wf[0], list(wl.wf[1]))], tag_rule=wl.rule)


def host_threads():
    """Host threads the CPU arm may use (torchrun exports OMP_NUM_THREADS=1: the oracle gets the count explicitly)."""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return max(1, os.cpu_count() or 1)


def oracle_run_jobs(oracle, op, wl, job_ids, n_threads=0, collect=None):
    """The CPU restatement on a set of jobs; returns (anchor pairs, seconds, walk steps, env members); the per-anchor
    scores of every job are appended to `collect` when given."""
    pairs, steps, members = 0, 0, 0
    t0 = time.perf_counter()
    for j in job_ids:
        a, b, anchors = wl.job_arrays(j)
        r = oracle.from_primitives(op, a.xyz, a.cat, a.tag, b.xyz, b.cat, b.tag, anchors, wl.threshold,
                                   n_threads=n_threads, debug=True)
        pairs += len(anchors)
        steps += int(r["steps"].sum())
        members += int(r["env_sizes"].sum())
        if collect is not None:
            collect.append(r["scores"])
    return pairs, time.perf_counter() - t0, steps, members


def other_workload(name, args, ctx, local_rank, fp64_peak):
    """One short run of another BASELINE configuration (N = 1 only): the `other_workloads` entry of the line."""
    xa = argparse.Namespace(**vars(args))
    if name == "cfg5":
        xa.ensemble = 96
    w2 = make_workload(name, 0, 1, xa)
    steps = max(3, min(args.steps, 5))
    r = measure(w2, ctx, local_rank, Solo(), steps, 3, args, clocks=False)
    tot = max(sum(v[0] for v in r["prof"].values()), 1e-9)
    return {"workload": w2.desc, "value": r["value"], "unit": "anchor-pairs/s",
            "ms_per_step": r["step_ms"], "anchor_pairs_per_step": w2.n_pairs,
            "e2e": r["e2e"], "gpu_launches": r["launches"],
            "kernel_ms_per_step": {g: ms / steps for g, (ms, n) in r["prof"].items() if n},
            "kernel_share": {g: ms / tot for g, (ms, n) in r["prof"].items() if n},
            "roofline_step_frac_fp64": (r["f_walk"] + r["f_gather"]) / (r["step_ms"] * 1e-3) / 1e12 / fp64_peak,
            "env_size_mean": float(r["sizes"].mean())}


def sample_parity(wl, ids, cpu_scores, gpu_results, means_only):
    """max |CPU - GPU| over the jobs `ids` (the first len(ids) jobs of the step, as sample_jobs returns them):
    cpu_scores[k] = the oracle's per-anchor scores of job ids[k]; gpu_results = the job means of the step (means_only)
    or its per-anchor scores, job after job.  nan if the GPU results do not cover the sample."""
    try:
        if means_only:
            return max(abs(float(sc.mean()) - float(gpu_results[j])) for j, sc in zip(ids, cpu_scores))
        offs = np.concatenate([[0], np.cumsum(wl.jobs["n"][:len(ids)])]).astype(np.int64)
        if offs[-1] > len(gpu_results):
            return float("nan")
        return max(float(np.abs(sc - gpu_results[offs[k]:offs[k + 1]]).max()) for k, sc in enumerate(cpu_scores))
    except (IndexError, ValueError):
        return float("nan")


def sample_jobs(wl, target_pairs):
    ids, tot = [], 0
    for j in range(len(wl.jobs)):
        ids.append(j)
        tot += int(wl.jobs["n"][j])
        if tot >= target_pairs:
            break
    return ids


def run_reference(args, rank, world):
    """--impl reference: the reference's algorithm on the host cores (oracle/, C++/OpenMP restatement)."""
    if rank != 0:
        return
    import oracle

    oracle.build()
    wl = make_workload(args.workload, 0, world, args)
    op = oracle_params(oracle, wl)
    ids = sample_jobs(wl, args.ref_pairs)
    cores = host_threads()
    for _ in range(args.warmup):
        oracle_run_jobs(oracle, op, wl, ids[:1], n_threads=cores)
    t, pairs = 0.0, 0
    for _ in range(args.steps):
        p, dt, _, _ = oracle_run_jobs(oracle, op, wl, ids, n_threads=cores)
        t += dt
        pairs += p
    value = pairs / t
    sample = f"{len(ids)} structure pair(s) = {pairs // max(args.steps, 1)} anchor pairs per step of workload {wl.name}"
    print(json.dumps({
        "impl": "reference", "metric": "anchor_pairs_per_second", "value": value, "unit": "anchor-pairs/s",
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * t / max(args.steps, 1),
        "higher_is_better": True, "scaling": wl.scaling, "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": wl.desc, "host": "CPU only"},
        "cpu_baseline": {"value": value, "unit": "anchor-pairs/s", "cores": cores, "kind": "port", "sample": sample,
                         "note": "C++/OpenMP restatement of the reference algorithm (kd-tree query, stable sort, "
                                 "sequential merge walk, pow-based Hellinger); the Rust crate cannot be built here"},
        "e2e": {"value": value, "unit": "anchor-pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }))


# ------------------------------------------------------------------------------------------------- GPU arm
def quiet_stdout():
    """stdout carries exactly one JSON line.  Libraries write to file descriptor 1 behind Python's back (NCCL prints its
    version banner there when the first communicator is created), so fd 1 is pointed at stderr for the run and the line
    is written to the saved descriptor at the end."""
    sys.stdout.flush()
    saved = os.dup(1)
    os.dup2(2, 1)
    return saved


def emit(saved_fd, text):
    sys.stdout.flush()
    os.write(saved_fd, (text + "\n").encode())


class Ranks:
    """Barrier / reductions over the ranks of the launch (no-ops for one process).  torch.distributed over NCCL is
    the benchmark's plumbing only: the scoring path has no collective."""

    def __init__(self, world, local_rank):
        import torch

        self.world, self.torch, self.dist = world, torch, None
        if world > 1:
            import torch.distributed as dist

            dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
            self.dist = dist

    def barrier(self):
        if self.dist:
            self.dist.barrier()

    def _reduce(self, x, op):
        if not self.dist:
            return x
        t = self.torch.tensor([x], dtype=self.torch.float64, device="cuda")
        self.dist.all_reduce(t, op=op)
        return float(t.item())

    def max(self, x):
        return self._reduce(x, self.dist.ReduceOp.MAX) if self.dist else x

    def sum(self, x):
        return self._reduce(x, self.dist.ReduceOp.SUM) if self.dist else x

    def close(self):
        if self.dist:
            self.dist.destroy_process_group()


class Solo:
    """The same interface for measurements that one rank makes on its own."""
    world = 1

    def barrier(self):
        pass

    def max(self, x):
        return x

    def sum(self, x):
        return x


def measure(wl, ctx, local_rank, ranks, steps, warmup, args, clocks=True):
    """Times `steps` passes of the hot path over workload `wl` with resident inputs (CUDA events on the library
    stream, max over ranks) and through host buffers (e2e); returns the numbers and the algorithmic work counts."""
    import torch

    from loco_hd_b200 import _capi

    ctx.set_params(wl.C, [wl.wf], tag_rule=wl.rule)
    stream = torch.cuda.ExternalStream(ctx.stream, device=torch.device("cuda", local_rank))
    n_env = len(wl.anchor_prim)

    # ---- resident inputs: structures in HBM (locohd_structs), anchors and outputs as device arrays
    structs = ctx.structs_create(wl.offsets, wl.xyz, wl.cat, wl.tag)
    d_as = torch.from_numpy(wl.anchor_struct.view(np.int32)).cuda()
    d_ap = torch.from_numpy(wl.anchor_prim.view(np.int32)).cuda()
    # The ensemble (and anything above --score-cap anchor pairs per step) returns only the per-job (= per structure
    # pair) means (SURVEY 8(f) N4, what compare_ensembles.py:293-299 computes next): the 1000-structure ensemble has
    # 2.5e9 anchor pairs = 20 GB of scores per step.  The per-anchor scores still exist (device scratch).
    means_only = wl.means_only or wl.n_pairs > args.score_cap
    n_out = len(wl.jobs) if means_only else wl.n_pairs
    d_out = torch.empty(n_out, dtype=torch.float64, device="cuda")

    def score(c, env, out):
        if means_only:
            c.score_jobs(env, env, wl.jobs, want_scores=False, means_out=out)
        else:
            c.score_jobs(env, env, wl.jobs, out=out)

    def step_resident():
        structs.drop_cells()  # the reference rebuilds its kd-trees on every call (locohd.rs:504-510): so do we
        env = ctx.envset_build(structs, d_ap.data_ptr(), wl.threshold, anchor_struct=d_as.data_ptr(), n_anchors=n_env)
        score(ctx, env, d_out.data_ptr())
        env.close()

    sampler = ClockSampler(local_rank) if clocks else None
    for _ in range(warmup):
        step_resident()
    ctx.synchronize()
    ctx.profile_read()
    ranks.barrier()
    torch.cuda.synchronize()
    t_begin = time.perf_counter()
    ctx.profile_enable(True)
    launches0 = ctx.launch_count
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(steps):
        step_resident()
    e1.record(stream)
    torch.cuda.synchronize()
    t_end = time.perf_counter()
    ranks.barrier()
    ms_total = ranks.max(e0.elapsed_time(e1))
    launches = ctx.launch_count - launches0
    prof = ctx.profile_read()
    ctx.profile_enable(False)
    clock_info = sampler.stop(t_begin, t_end) if sampler else None
    total_pairs = ranks.sum(float(wl.n_pairs))
    value = total_pairs * steps / (ms_total * 1e-3)

    # ---- algorithmic work (SURVEY.md §8(d)) from the environment sizes of one extra, untimed build
    env = ctx.envset_build(structs, d_ap.data_ptr(), wl.threshold, anchor_struct=d_as.data_ptr(), n_anchors=n_env)
    off = np.empty(n_env + 1, np.uint64)
    ctx._check(ctx.lib.locohd_envset_dump(ctx.h, env.h, _capi._p(off), None, None, None))
    check_scores = d_out.cpu().numpy()
    env.close()
    structs.close()
    del d_out
    sizes = np.diff(off).astype(np.int64)
    ja, jb, jn = (wl.jobs[k].astype(np.int64) for k in ("a_first", "b_first", "n"))
    members = (off[ja + jn] - off[ja]).astype(np.int64) + (off[jb + jn] - off[jb]).astype(np.int64)  # sum of Ma + Mb per job
    events = members - jn                                    # sum of E = Ma + Mb - 1 (cross-list exact ties: none here)
    f_walk = float(events.sum()) * (10 * wl.C + 4 + F_WF[wl.wf[0]])
    f_gather = float(10 * sizes.sum())                       # every environment is gathered once per step
    alg_bytes = 16.0 * wl.n_pairs + 29.0 * float(wl.offsets[-1])

    # ---- e2e: host (pinned) buffers through the same C-ABI calls, copies inside the timed region
    h_off = wl.offsets
    h_xyz = ctx.pinned_array(wl.xyz.shape, np.float64); h_xyz[...] = wl.xyz
    h_cat = ctx.pinned_array(wl.cat.shape, np.uint16); h_cat[...] = wl.cat
    h_tag = ctx.pinned_array(wl.tag.shape, np.uint32); h_tag[...] = wl.tag
    h_as = ctx.pinned_array(wl.anchor_struct.shape, np.uint32); h_as[...] = wl.anchor_struct
    h_ap = ctx.pinned_array(wl.anchor_prim.shape, np.uint32); h_ap[...] = wl.anchor_prim
    h_out = ctx.pinned_array((n_out,), np.float64)

    # One upload at a time: with two host threads the lock puts them in anti-phase by itself (one uploads its step
    # while the other one's kernels run) instead of both copying, then both computing.
    upload_lock = threading.Lock()

    def step_e2e(c=ctx, out=h_out, xyz=h_xyz):
        with upload_lock:
            st = c.structs_create(h_off, xyz, h_cat, h_tag)
        env = c.envset_build(st, h_ap, wl.threshold, anchor_struct=h_as)
        score(c, env, out)
        env.close()
        st.close()

    step_ms = ms_total / steps
    long_steps = step_ms > 500.0            # seconds-long steps: copies are noise, two timed steps are enough
    e2e_steps = 2 if long_steps else 6
    for _ in range(1 if long_steps else 2):
        step_e2e()
    ctx.synchronize()
    ranks.barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        step_e2e()
    ctx.synchronize()
    t_serial = ranks.max(time.perf_counter() - t0)
    e2e_serial = total_pairs * e2e_steps / t_serial
    e2e_ok = bool(np.array_equal(h_out, check_scores))
    e2e = {"value": e2e_serial, "unit": "anchor-pairs/s", "h2d_bytes_per_step": int(wl.h2d_bytes),
           "d2h_bytes_per_step": int(8 * n_out), "steps": e2e_steps, "mode": "one host thread, steps back to back",
           "one_thread_value": e2e_serial}

    if not long_steps:
        # The same calls from two (LOCOHD_BENCH_E2E_THREADS) host threads, each with its own context (= stream) and
        # output buffer: the H2D copies of one step overlap the kernels of the other.  Every step still uploads its
        # inputs from pinned host memory and reads its scores back inside the timed region.
        n_thr = max(2, int(os.environ.get("LOCOHD_BENCH_E2E_THREADS", "2")))
        extra = []
        for _ in range(n_thr - 1):
            c = _capi.Context(local_rank)
            c.set_params(wl.C, [wl.wf], tag_rule=wl.rule)
            extra.append((c, c.pinned_array((n_out,), np.float64)))
        lanes = [(ctx, h_out)] + extra
        pipe_steps = 12 // n_thr * n_thr       # enough steps per thread to amortise the fill and drain of the pipeline

        def run_pipelined(n_each, xyz):
            def worker(c, out):
                torch.cuda.set_device(local_rank)
                for _ in range(n_each):
                    step_e2e(c, out, xyz)
                c.synchronize()

            ths = [threading.Thread(target=worker, args=lane) for lane in lanes]
            for t in ths:
                t.start()
            for t in ths:
                t.join()

        def timed_pipeline(xyz):
            run_pipelined(1, xyz)
            ranks.barrier()
            t0 = time.perf_counter()
            run_pipelined(pipe_steps // n_thr, xyz)
            return total_pairs * pipe_steps / ranks.max(time.perf_counter() - t0)

        e2e_pipe = timed_pipeline(h_xyz)
        e2e_ok = e2e_ok and all(bool(np.array_equal(o, check_scores)) for _, o in extra)
        e2e["two_thread_value"] = e2e_pipe
        e2e["pipelined"] = {"host_threads": n_thr, "steps": pipe_steps}
        if e2e_pipe > e2e_serial:
            e2e["value"], e2e["steps"] = e2e_pipe, pipe_steps
            e2e["mode"] = f"{n_thr} host threads / contexts, copies of one step overlap kernels of the other"

        # f32 wire format (locohd_structs_create_f32): real coordinates are float32 (Bio.PDB, MDAnalysis), the synthetic
        # ones are rounded through float32 for this variant only; half the coordinate bytes cross the bus.  Reported
        # beside the f64 figure, not instead of it (different inputs).
        if wl.name in ("cfg3", "cfg4"):
            x32 = ctx.pinned_array(wl.xyz.shape, np.float32); x32[...] = wl.xyz
            e2e["f32_wire"] = {"value": timed_pipeline(x32), "mode": f"{n_thr} host threads / contexts",
                               "h2d_bytes_per_step": int(wl.h2d_bytes - wl.xyz.nbytes // 2),
                               "note": "coordinates rounded through float32 and uploaded as float32 (exact widening on the device)"}
        for c, _ in extra:
            c.close()
    e2e["scores_identical_to_resident_run"] = e2e_ok

    return {"value": value, "ms_total": ms_total, "step_ms": step_ms, "launches": int(launches), "prof": prof,
            "clocks": clock_info, "total_pairs": total_pairs, "n_env": n_env, "sizes": sizes, "f_walk": f_walk,
            "f_gather": f_gather, "alg_bytes": alg_bytes, "check_scores": check_scores, "means_only": means_only,
            "e2e": e2e, "n_out": n_out}


def python_api_latency(local_rank):
    """The drop-in Python API on single structure pairs (what a user of the reference calls): LoCoHD.from_primitives
    with lists of PrimitiveAtom / anchor tuples, and the array form from_arrays, against the bare C-ABI call."""
    import loco_hd
    from loco_hd_b200 import _capi

    loco_hd.loco_hd.set_device(local_rank)
    out = {}
    ctx = _capi.Context(local_rank)
    for key, (a, b), C, wf, step in (("cfg1_150_anchors", synth.config1(), 7, ("uniform", (3.0, 10.0)), 3),
                                     ("cfg2_10000_anchors", synth.config2(), 7, ("kumaraswamy", (3.0, 10.0, 2.0, 5.0)), 1)):
        anchors = np.stack([np.arange(0, a.n, step, dtype=np.uint32)] * 2, axis=1)
        ctx.set_params(C, [wf], tag_rule={"accept_same": False})
        lchd = loco_hd.LoCoHD([f"T{i}" for i in range(C)], loco_hd.WeightFunction(wf[0], list(wf[1])),
                              loco_hd.TagPairingRule({"accept_same": False}))
        pa = [loco_hd.PrimitiveAtom(f"T{c}", str(t), x) for x, c, t in zip(a.xyz.tolist(), a.cat, a.tag)]
        pb = [loco_hd.PrimitiveAtom(f"T{c}", str(t), x) for x, c, t in zip(b.xyz.tolist(), b.cat, b.tag)]
        ap = [tuple(map(int, q)) for q in anchors]
        calls = {"c_abi": lambda: ctx.from_primitives(a.xyz, a.cat, a.tag, b.xyz, b.cat, b.tag, anchors, 10.0),
                 "from_primitives_lists": lambda: lchd.from_primitives(pa, pb, ap, 10.0),
                 "from_arrays": lambda: lchd.from_arrays(a.xyz, a.cat, a.tag, b.xyz, b.cat, b.tag, anchors, 10.0)}
        row = {}
        ref = None
        for name, fn in calls.items():
            for _ in range(3):
                r = np.asarray(fn())
            n = 20
            t0 = time.perf_counter()
            for _ in range(n):
                fn()
            dt = (time.perf_counter() - t0) / n
            ref = r if ref is None else ref
            row[name] = {"ms_per_call": 1e3 * dt, "anchor_pairs_per_s": len(anchors) / dt,
                         "identical_to_c_abi": bool(np.array_equal(r, ref))}
        out[key] = row
    ctx.close()
    return out


DUMP_BYTES = 64 << 20


def dump_outputs(out_dir, result, means_only, rank, world):
    """--dump-outputs: what the last timed step handed to its caller (the per-structure-pair means, or the per-anchor
    scores), float64, as OUT_DIR/<name>.npy; one file per rank when several run.  Above 64 MB in all, the values at a
    fixed set of positions (seeded, sorted) are written instead, as <name>_sample.npy, so that two builds run with the
    same arguments can still be compared value for value."""
    name = ("job_means" if means_only else "scores") + (f"_rank{rank}" if world > 1 else "")
    result = np.asarray(result, dtype=np.float64)
    cap = DUMP_BYTES // (8 * world)
    if len(result) > cap:
        result = result[np.unique(np.random.default_rng(0).integers(0, len(result), size=cap))]
        name += "_sample"
    out = Path(out_dir)
    out.mkdir(parents=True, exist_ok=True)
    np.save(out / f"{name}.npy", result)
    return out / f"{name}.npy"


def run_gpu(args, rank, local_rank, world):
    stdout_fd = quiet_stdout()
    _ensure_built()
    import torch

    from loco_hd_b200 import _capi

    torch.cuda.set_device(local_rank)
    ranks = Ranks(world, local_rank)
    wl = make_workload(args.workload, rank, world, args)
    if args.threshold:   # exploration only: the BASELINE configurations use 10 A
        wl.threshold = float(args.threshold)
        wl.desc += f" [threshold overridden: {wl.threshold:g}]"
    ctx = _capi.Context(local_rank)
    m = measure(wl, ctx, local_rank, ranks, args.steps, args.warmup, args)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, m["check_scores"], m["means_only"], rank, world)
    if rank != 0:
        ctx.close()
        ranks.close()
        return
    prof, sizes, step_ms = m["prof"], m["sizes"], m["step_ms"]
    f_walk, f_gather, alg_bytes, means_only = m["f_walk"], m["f_gather"], m["alg_bytes"], m["means_only"]

    # ---- rooflines (rank 0's kernels; all ranks run identical shapes)
    peaks = {}
    try:
        peaks = json.loads((ROOT / "MEASURED_PEAKS.json").read_text())
    except OSError:
        pass
    hbm_peak, hbm_src = (peaks["hbm_gbs"], "measured (MEASURED_PEAKS.json)") if "hbm_gbs" in peaks else (6650.0, "fallback")
    probe_clocks = ClockSampler(local_rank)
    t_p0 = time.perf_counter()
    fp64_peak = ctx.measure_fp64_tflops()
    probe_info = probe_clocks.stop(t_p0, time.perf_counter())
    kernels = {g: {"ms_per_step": ms / args.steps, "share": ms / max(sum(v[0] for v in prof.values()), 1e-9)}
               for g, (ms, n) in prof.items() if n}
    # Algorithmic flops per kernel (SURVEY.md 8(d)): walk E * (10 C + 4 + F_wf) -> K2; the 10 flops per environment
    # member (3 sub, 3 mul, 2 add, 1 compare, 1 sqrt) all belong to the fused gather K1; the sampled upper-bound
    # pass does no algorithmic FP64 work.  With LOCOHD_LEGACY_GATHER=1 the multi-kernel path runs instead (9 of the
    # 10 in the exact fill K1b, the sqrt in the sort K1c).
    score_name = ("score_tile_kernel (K2t: merge walk per 4x4 tile of structure pairs, 8 environments staged per 16 anchor pairs)"
                  if ctx.tile_launches else "score_fast_kernel / score_kernel (K2 merge walk)")
    if "sort" in kernels:
        alg = {"score": (score_name, f_walk),
               "fill": ("env_tile_kernel<true> (K1b exact gather, multi-kernel path)", 0.9 * f_gather),
               "sort": ("env_sort_kernel (K1c sort + CDF + packing, multi-kernel path)", 0.1 * f_gather),
               "count": ("env_tile_kernel<false> (K1a FP32 upper-bound sizes)", 0.0)}
    else:
        alg = {"score": (score_name, f_walk),
               "fill": ("env_fused_kernel (K1: row pruning, exact FP64 gather, register bitonic sort, CDF, packing)",
                        f_gather),
               "count": ("env_tile_kernel<false> with stride 16 (store sizing sample)", 0.0)}
    traffic, pipes, prof_src, traffic_note = {}, {}, None, None
    for tf in sorted((ROOT / "profiles").glob("*_traffic.json"), reverse=True):   # newest round first
        try:
            tr = json.loads(tf.read_text())
        except (OSError, ValueError):
            continue
        if tr.get("workload") == wl.name and tr.get("anchor_pairs_per_step") == wl.n_pairs:
            traffic = tr.get("dram_bytes_per_launch", {})
            pipes = tr.get("pipes", {})
            prof_src = tr.get("source")
            traffic_note = tr.get("note")
            break
    per_kernel = {}
    for g, (name, flops) in alg.items():
        if g in kernels and kernels[g]["ms_per_step"] > 0:
            ach = flops / (kernels[g]["ms_per_step"] * 1e-3) / 1e12
            per_kernel[g] = {"kernel": name, "launch_ms": kernels[g]["ms_per_step"], "alg_flops_per_launch": flops,
                             "achieved_tflops": ach, "frac_of_fp64_peak": ach / fp64_peak, "traffic": traffic.get(g)}
            if g in pipes:   # from the committed ncu capture of the same workload (not measured in this run)
                per_kernel[g]["ncu"] = dict(pipes[g], source=prof_src)
                wf = pipes[g].get("shared_wavefronts")
                if wf and probe_info.get("sm_mhz"):
                    # the pipe that binds the scoring kernels: one shared-memory wavefront per clock and SM; wavefronts
                    # per launch from the committed ncu capture, launch time and SM clock measured in this run
                    peak_wf = 148 * probe_info["sm_mhz"] * 1e6
                    ach_wf = wf / (kernels[g]["ms_per_step"] * 1e-3)
                    per_kernel[g]["shared_pipe_roofline"] = {
                        "bound": "shared-memory data pipe (1 wavefront / clock / SM)", "achieved": ach_wf / 1e9,
                        "peak": peak_wf / 1e9, "unit": "G wavefronts/s", "frac": ach_wf / peak_wf,
                        "wavefronts_per_launch": wf, "bank_conflict_share": (pipes[g].get("shared_bank_conflicts") or 0) / wf}
    dom = max(per_kernel, key=lambda g: per_kernel[g]["launch_ms"])
    dominant, dom_flops, dom_ms = per_kernel[dom]["kernel"], per_kernel[dom]["alg_flops_per_launch"], per_kernel[dom]["launch_ms"]
    achieved = dom_flops / (dom_ms * 1e-3) / 1e12
    roofline = {
        "kernel": dominant,
        "bound": "fp64", "achieved": achieved, "peak": fp64_peak, "unit": "TFLOP/s", "frac": achieved / fp64_peak,
        "peak_source": (f"FP64 FMA probe kernel run in this process: {fp64_peak:.2f} TFLOP/s at SM "
                        f"{probe_info.get('sm_mhz')} MHz (max {probe_info.get('sm_max_mhz')}), reasons "
                        f"{probe_info.get('reasons')}; MEASURED_PEAKS.json has no FP64 entry (nominal 148 SM x 64 FMA/clk "
                        "x 2 x 1.965 GHz = 37.2)"),
        "peak_probe": {"tflops": fp64_peak, "clocks": probe_info},
        "traffic": traffic.get(dom), "alg_flops_per_launch": dom_flops, "launch_ms": dom_ms,
        "note": "traffic = dram__bytes_read.sum + dram__bytes_write.sum of one launch from profiles/ (ncu)"
                + (f"; {traffic_note}" if traffic_note else ""),
    }
    roofline_hbm = {"bound": "hbm", "achieved": alg_bytes / (step_ms * 1e-3) / 1e9, "peak": hbm_peak, "unit": "GB/s",
                    "frac": alg_bytes / (step_ms * 1e-3) / 1e9 / hbm_peak, "peak_source": hbm_src,
                    "alg_bytes_per_step": alg_bytes, "scope": "whole step"}
    roofline_step = {"bound": "fp64", "achieved": (f_walk + f_gather) / (step_ms * 1e-3) / 1e12, "peak": fp64_peak,
                     "unit": "TFLOP/s", "frac": (f_walk + f_gather) / (step_ms * 1e-3) / 1e12 / fp64_peak,
                     "scope": "whole step (ALG_FLOPS of SURVEY.md 8(d))"}

    # ---- CPU baseline beside it (rank 0, N = 1 only): the oracle on a bounded sample of the same workload
    cpu = None
    check_scores = m["check_scores"]
    if world == 1 and not args.no_cpu_baseline:
        try:
            import oracle

            oracle.build()
            op = oracle_params(oracle, wl)
            ids = sample_jobs(wl, args.cpu_pairs)   # ~10 s of CPU work on 16 threads
            cores = host_threads()
            oracle_run_jobs(oracle, op, wl, ids[:1], n_threads=cores)
            cpu_scores = []
            p, dt, steps, members = oracle_run_jobs(oracle, op, wl, ids, n_threads=cores, collect=cpu_scores)
            ids1 = sample_jobs(wl, max(1, args.ref_pairs // 16))
            p1, dt1, _, _ = oracle_run_jobs(oracle, op, wl, ids1, n_threads=1)
            # the sample doubles as a parity spot check of this very run
            a, b, anchors = wl.job_arrays(0)
            ref = oracle.from_primitives(op, a.xyz, a.cat, a.tag, b.xyz, b.cat, b.tag, anchors, wl.threshold)
            n0 = int(wl.jobs["n"][0])
            # ... and every job of the timed sample against this run's GPU results (on the default workload: the first 200
            # structure pairs = 13 tiles, all 5000 anchors of each, i.e. every anchor slice of the tile kernel's unit order)
            sample_diff = sample_parity(wl, ids, cpu_scores, check_scores, means_only)
            cpu = {"value": p / dt, "unit": "anchor-pairs/s", "cores": cores, "kind": "port",
                   "sample": f"first {len(ids)} structure pair(s) of the step = {p} anchor pairs, {dt:.2f} s",
                   "single_thread_value": p1 / dt1,
                   "walk_steps_per_pair": steps / p, "env_members_per_pair": members / p,
                   ("max_abs_mean_score_diff_vs_gpu_job0" if means_only else "max_abs_score_diff_vs_gpu_job0"):
                       float(abs(ref.mean() - check_scores[0]) if means_only else np.abs(ref - check_scores[:n0]).max()),
                   ("max_abs_mean_score_diff_vs_gpu_sample" if means_only else "max_abs_score_diff_vs_gpu_sample"): sample_diff,
                   "note": "C++/OpenMP restatement of the reference algorithm (Rust toolchain unavailable)"}
        except Exception as exc:   # an optional section must not cost the headline line
            cpu = {"error": repr(exc), "kind": "port"}

    # ---- the other BASELINE configurations, one short run each (N = 1 only), and the Python API
    others, py_api = None, None
    if world == 1 and not args.no_extras:
        others = {}
        for name in ("cfg2", "cfg3", "cfg4", "cfg5"):
            if name == wl.name:
                continue
            try:
                others[name] = other_workload(name, args, ctx, local_rank, fp64_peak)
            except Exception as exc:   # an optional section must not cost the headline line
                others[name] = {"error": repr(exc)}
        try:
            py_api = python_api_latency(local_rank)
        except Exception as exc:
            py_api = {"error": repr(exc)}

    line = {
        "metric": "anchor_pairs_per_second", "value": m["value"], "unit": "anchor-pairs/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": step_ms, "higher_is_better": True,
        "scaling": wl.scaling, "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": wl.desc, "anchor_pairs_per_gpu_per_step": wl.n_pairs,
                   "anchor_pairs_per_step_all_gpus": int(m["total_pairs"]),
                   "environments_per_gpu_per_step": m["n_env"],
                   "result": ("per-structure-pair mean scores (locohd_score_jobs out_job_means); the per-anchor scores "
                              "stay in device scratch") if means_only else "per-anchor scores",
                   "l2": f"inputs larger than L2 each step: {wl.h2d_bytes / 1e6:.0f} MB of structures/anchors + "
                         f"{8 * float(sizes.sum()) / 1e6:.0f} MB environment store written per step and streamed by K2"},
        "e2e": m["e2e"],
        "gpu_launches": m["launches"],
        "clocks": m["clocks"],
        "roofline": roofline, "roofline_hbm": roofline_hbm, "roofline_step": roofline_step,
        "kernels": kernels, "kernel_rooflines": per_kernel,
        "env_size_mean": float(sizes.mean()), "env_size_max": int(sizes.max()),
        "cpu_baseline": cpu,
        "other_workloads": others,
        "e2e_python": py_api,
    }
    emit(stdout_fd, json.dumps(line))
    ctx.close()
    ranks.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="cfg5", choices=["cfg2", "cfg3", "cfg4", "cfg5"])
    ap.add_argument("--pairs", type=int, default=256, help="cfg2: structure pairs per GPU per step")
    ap.add_argument("--models", type=int, default=500, help="cfg3: models per GPU per step")
    ap.add_argument("--frames", type=int, default=1024, help="cfg4: frames per GPU per step")
    ap.add_argument("--ensemble", type=int, default=1000, help="cfg5: ensemble size (all-vs-all, jobs dealt over GPUs)")
    ap.add_argument("--ref-pairs", type=int, default=160000, help="anchor pairs per step of the CPU reference arm")
    ap.add_argument("--cpu-pairs", type=int, default=1000000, help="anchor pairs of the cpu_baseline sample of the GPU arm")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the short runs of the other configurations and the Python-API latencies")
    ap.add_argument("--score-cap", type=int, default=1 << 28,
                    help="above this many anchor pairs per GPU per step only the per-job means are copied out")
    ap.add_argument("--threshold", type=float, default=0.0, help="override the 10 A threshold (exploration only)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the results of the last one to DIR/<name>.npy (float64, at most "
                         "64 MB in all; a fixed seeded sample of larger results)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the GPU path's results; the reference arm has none")
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world != args.gpus and world == 1 and args.gpus > 1:
        # launched without torchrun: re-launch one process per GPU
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}",
               "--master-addr", "127.0.0.1", "--master-port", "29517", str(Path(__file__).resolve())] + sys.argv[1:]
        raise SystemExit(subprocess.call(cmd))
    if args.impl == "reference":
        run_reference(args, rank, world)
    else:
        run_gpu(args, rank, local_rank, world)


if __name__ == "__main__":
    main()
