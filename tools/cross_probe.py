"""Cost of cross matrices (locohd_score_cross) against the routes a caller had before it, on one GPU.

Environments of configuration-5-like structures (5000 primitives, C = 7, uniform [3, 10], 10 A, hetero contacts, every
primitive an anchor): 21 structures in one env-set, A = the 5000 environments of structure 0, B = those of the others.
Shapes:
  * 2 000 x 50 000: score_cross (tile route, LOCOHD_NO_TILES=1 pair route; scores to host memory as score_matrix
    returns them, and to a device matrix), score_pairs on the explicit pair list (host list, host scores);
  * 400 x 5 000 (2 x 10^6 one-anchor jobs, a 48 MB job table): score_cross against score_batch with one-anchor jobs in
    4 x 4 blocked order;
  * 1 x 10 000 (kras_scan.py:47-52): score_cross on both routes, score_pairs, score_batch;
  * 5 000 x 100 000 k nearest (k = 16, matrix kept on the device) and the device memory that call takes at its peak
    (cudaMemGetInfo sampled every millisecond from a second thread while the call runs, above the value before
    the context's first scoring call).
  * condensed vectors of one range (locohd_score_condensed) against score_cross of the range against itself, the two
    calls alternated rep by rep: the first 20 000 environments into device and into host memory, the first 50 000
    into device memory only (a 20 GB matrix), each on the tile route and the LOCOHD_NO_TILES=1 pair route; the
    vector is checked bit for bit against the matrix's strict upper triangle on the device.
  * threshold graphs (locohd_score_within[_condensed], names starting with "within"), alternated with the dense calls
    they replace: 2 000 x 50 000 on both routes at max_score = the 0.1 %, 10 % and 100 % quantiles of that matrix,
    the graph kept on the device against score_cross into a device matrix, and the graph copied to host arrays (what
    LoCoHD.environments_within returns) against score_cross into host memory (score_matrix); the first 20 000
    environments in within mode against score_condensed into device and host memory.  Every graph is checked bit for
    bit against the thresholded dense result.
Times are host clocks around whole calls (each ends in a device synchronisation): median of --reps after --warmup.
The card's name and power limit are read in the same run.  Prints one JSON line per measurement, appends them to --out.
--lib runs against another build of the library (the A/B of the kernel's unit order); --only restricts to names
containing that string.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np

ap = argparse.ArgumentParser()
ap.add_argument("--reps", type=int, default=5)
ap.add_argument("--warmup", type=int, default=1)
ap.add_argument("--out", default=None)
ap.add_argument("--lib", default=None)
ap.add_argument("--label", default="main")
ap.add_argument("--only", default="")
args = ap.parse_args()
if args.lib:
    os.environ["LOCOHD_LIB"] = args.lib

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
import torch  # noqa: E402

from benchdata import synth  # noqa: E402
from loco_hd_b200 import _capi  # noqa: E402

GPU = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                     text=True).stdout.strip().splitlines()[0]
N_STRUCT, PER = 21, 5000


def emit(rec):
    rec = {"gpu": GPU, "lib": args.label, **rec}
    line = json.dumps(rec)
    print(line, flush=True)
    if args.out:
        with open(args.out, "a") as f:
            f.write(line + "\n")


def timed(name, pairs, f):
    if args.only not in name:
        return
    for _ in range(args.warmup):
        f()
    t = []
    for _ in range(args.reps):
        t0 = time.perf_counter()
        f()
        t.append(time.perf_counter() - t0)
    med = float(np.median(t))
    emit({"name": name, "pairs": int(pairs), "ms": round(1e3 * med, 3), "ms_min": round(1e3 * min(t), 3),
          "ms_max": round(1e3 * max(t), 3), "pairs_per_s": pairs / med})


def blocked_jobs(a0, n_a, b0, n_b):
    """One-anchor jobs (a0 + i, b0 + j, 1) listed in 4 x 4 blocks: what locohd_score_jobs tiles."""
    i, j = np.meshgrid(np.arange(n_a), np.arange(n_b), indexing="ij")
    order = np.lexsort(((j % 4).ravel(), (i % 4).ravel(), (j // 4).ravel(), (i // 4).ravel()))
    jobs = np.zeros(n_a * n_b, dtype=_capi.JOB_DTYPE)
    jobs["a_first"] = a0 + i.ravel()[order]
    jobs["b_first"] = b0 + j.ravel()[order]
    jobs["n"] = 1
    return jobs


def pair_list(a0, n_a, b0, n_b):
    i, j = np.meshgrid(np.arange(n_a) + a0, np.arange(n_b) + b0, indexing="ij")
    return np.stack([i.ravel(), j.ravel()], axis=1).astype(np.uint32)


def main():
    torch.cuda.init()
    ctx = _capi.Context(0)
    ctx.set_params(7, [("uniform", (3.0, 10.0))], tag_rule={"accept_same": False})
    base = synth.config5_base()
    clouds = [synth.config5_member(base, i) for i in range(N_STRUCT)]
    offs = np.cumsum([0] + [c.n for c in clouds]).astype(np.uint64)
    st = ctx.structs_create(offs, np.concatenate([c.xyz for c in clouds]), np.concatenate([c.cat for c in clouds]),
                            np.concatenate([c.tag for c in clouds]))
    anchors = np.arange(PER, dtype=np.uint32)
    env = ctx.envset_build(st, np.tile(anchors, N_STRUCT), 10.0,
                           anchor_struct=np.repeat(np.arange(N_STRUCT, dtype=np.uint32), PER))
    geo = _capi.tile_geometry(7, 1024, 1024)
    emit({"name": "setup", "environments": len(env), "members": env.total_members, "tile_geometry_1024": geo})

    def cross(n_a, n_b, **kw):
        return lambda: ctx.score_cross(env, env, 0, n_a, PER, n_b, **kw)

    # 5 000 x 100 000, k = 16, the matrix kept on the device
    name = "nearest_5000x100000_k16"
    if args.only in name:
        peak = [0]
        before, _ = torch.cuda.mem_get_info()
        done = threading.Event()

        def sample():
            while not done.is_set():
                free, _ = torch.cuda.mem_get_info()
                peak[0] = max(peak[0], before - free)
                time.sleep(0.001)

        th = threading.Thread(target=sample)
        th.start()
        timed(name, 5e8, cross(5000, 100_000, scores=False, k=16))
        done.set()
        th.join()
        emit({"name": name + "_memory", "peak_device_bytes_of_the_call": int(peak[0]),
              "store_bytes": int(env.total_members) * 8, "note": "device use above the moment before the first call of the context that scores (the environment store is held before it)"})

    # 2 000 x 50 000
    dev = torch.empty((2000, 50_000), dtype=torch.float64, device="cuda")
    t0 = ctx.tile_launches
    timed("cross_2000x50000_tiles_host", 1e8, cross(2000, 50_000))
    emit({"name": "tile_launches_check", "tile_launches": ctx.tile_launches - t0})
    timed("cross_2000x50000_tiles_device", 1e8, cross(2000, 50_000, scores=dev.data_ptr()))
    if args.lib is None:
        ref = ctx.score_cross(env, env, 0, 2000, PER, 50_000)[0]
        os.environ["LOCOHD_NO_TILES"] = "1"
        timed("cross_2000x50000_pairs_host", 1e8, cross(2000, 50_000))
        timed("cross_2000x50000_pairs_device", 1e8, cross(2000, 50_000, scores=dev.data_ptr()))
        pr = ctx.score_cross(env, env, 0, 2000, PER, 50_000)[0]
        del os.environ["LOCOHD_NO_TILES"]
        emit({"name": "tiles_vs_pairs_2000x50000", "max_abs_diff": float(np.abs(ref - pr).max())})
        del ref, pr
        pl = pair_list(0, 2000, PER, 50_000)
        timed("score_pairs_2000x50000", 1e8, lambda: ctx.score_pairs(env, env, pl))
        del pl
    del dev
    if args.lib is not None:
        return

    # 400 x 5 000: score_batch's one-anchor jobs where the job table is modest
    jobs = blocked_jobs(0, 400, PER, 5000)
    timed("cross_400x5000_tiles_host", 2e6, cross(400, 5000))
    t0 = ctx.tile_launches
    timed("score_batch_blocked_400x5000", 2e6, lambda: ctx.score_jobs_stats(env, env, jobs, scores=True))
    emit({"name": "score_batch_tile_launches", "tile_launches": ctx.tile_launches - t0})

    # 1 x 10 000 (kras_scan)
    timed("cross_1x10000_tiles_host", 1e4, cross(1, 10_000))
    os.environ["LOCOHD_NO_TILES"] = "1"
    timed("cross_1x10000_pairs_host", 1e4, cross(1, 10_000))
    del os.environ["LOCOHD_NO_TILES"]
    pl = pair_list(0, 1, PER, 10_000)
    timed("score_pairs_1x10000", 1e4, lambda: ctx.score_pairs(env, env, pl))
    kj = blocked_jobs(0, 1, PER, 10_000)
    timed("score_batch_1x10000", 1e4, lambda: ctx.score_jobs_stats(env, env, kj, scores=True))

    within(ctx, env)
    condensed(ctx, env)
    env.close()
    st.close()


def alternated(name, a, b):
    """a, b: (label, pairs, f).  The two calls alternate rep by rep, so drifts of the shared host and clocks hit both."""
    if args.only not in name:
        return
    for _ in range(args.warmup):
        a[2]()
        b[2]()
    t = {a[0]: [], b[0]: []}
    for _ in range(args.reps):
        for label, _, f in (a, b):
            t0 = time.perf_counter()
            f()
            t[label].append(time.perf_counter() - t0)
    med = {k: float(np.median(v)) for k, v in t.items()}
    for label, pairs, _ in (a, b):
        emit({"name": f"{name}_{label}", "pairs": int(pairs), "ms": round(1e3 * med[label], 3),
              "ms_min": round(1e3 * min(t[label]), 3), "ms_max": round(1e3 * max(t[label]), 3),
              "pairs_per_s": pairs / med[label]})
    emit({"name": f"{name}_ratio", f"{a[0]}_over_{b[0]}": round(med[a[0]] / med[b[0]], 4)})


def graph_equals(g, indptr, indices, scores):
    ip, ix, sc = g.copy()
    return bool(np.array_equal(ip, indptr) and np.array_equal(ix, indices) and
                np.array_equal(sc.view(np.uint64), scores.view(np.uint64)))


def within(ctx, env):
    n_a, n_b = 2000, 50_000
    for route in ("tiles", "pairs"):
        name = f"within_2000x50000_{route}"
        if args.only not in name:
            continue
        if route == "pairs":
            os.environ["LOCOHD_NO_TILES"] = "1"
        M = ctx.score_cross(env, env, 0, n_a, PER, n_b)[0]
        dev = torch.empty((n_a, n_b), dtype=torch.float64, device="cuda")
        for q, bound in zip((0.001, 0.1, 1.0), np.quantile(M, (0.001, 0.1, 1.0))):
            bound = float(bound)
            t0 = ctx.tile_launches
            g = ctx.score_within(env, env, bound, 0, n_a, PER, n_b)
            keep = M <= bound
            r, c = np.nonzero(keep)
            indptr = np.concatenate([[0], np.cumsum(keep.sum(axis=1))]).astype(np.uint64)
            emit({"name": f"{name}_q{q}", "max_score": bound, "nnz": g.nnz, "density": g.nnz / (n_a * n_b),
                  "tile_launches": ctx.tile_launches - t0,
                  "bit_identical_to_thresholded_matrix": graph_equals(g, indptr, c.astype(np.uint32), M[r, c])})
            g.close()
            del keep, r, c
            alternated(f"{name}_q{q}_device",
                       ("graph", n_a * n_b, lambda: ctx.score_within(env, env, bound, 0, n_a, PER, n_b).close()),
                       ("matrix", n_a * n_b, lambda: ctx.score_cross(env, env, 0, n_a, PER, n_b, scores=dev.data_ptr())))

            def to_host():
                g = ctx.score_within(env, env, bound, 0, n_a, PER, n_b)
                g.copy()
                g.close()

            alternated(f"{name}_q{q}_host", ("graph", n_a * n_b, to_host),
                       ("matrix", n_a * n_b, lambda: ctx.score_cross(env, env, 0, n_a, PER, n_b)))
        del M, dev
        torch.cuda.empty_cache()
    os.environ.pop("LOCOHD_NO_TILES", None)
    n = 20_000
    name = f"within_condensed_{n}_tiles"
    if args.only not in name:
        return
    c = ctx.score_condensed(env, 0, n)
    k = [int(q * (len(c) - 1)) for q in (0.001, 0.1)]
    part = np.partition(c, k)
    vec = torch.empty(len(c), dtype=torch.float64, device="cuda")
    for q, bound in ((0.001, part[k[0]]), (0.1, part[k[1]]), (1.0, c.max())):
        bound = float(bound)
        g = ctx.score_within_condensed(env, bound, 0, n)
        iu, ju = np.triu_indices(n, 1)
        keep = c <= bound
        indptr = np.zeros(n + 1, np.uint64)
        indptr[1:] = np.cumsum(np.bincount(iu[keep], minlength=n))
        emit({"name": f"{name}_q{q}", "max_score": bound, "nnz": g.nnz, "density": g.nnz / len(c),
              "bit_identical_to_thresholded_condensed": graph_equals(g, indptr, ju[keep].astype(np.uint32), c[keep])})
        g.close()
        del iu, ju, keep
        alternated(f"{name}_q{q}_device",
                   ("graph", len(c), lambda: ctx.score_within_condensed(env, bound, 0, n).close()),
                   ("condensed", len(c), lambda: ctx.score_condensed(env, 0, n, out=vec.data_ptr())))

        def to_host():
            g = ctx.score_within_condensed(env, bound, 0, n)
            g.copy()
            g.close()

        alternated(f"{name}_q{q}_host", ("graph", len(c), to_host),
                   ("condensed", len(c), lambda: ctx.score_condensed(env, 0, n)))
    del c, part, vec
    torch.cuda.empty_cache()


def condensed(ctx, env):
    for route in ("tiles", "pairs"):
        if route == "pairs":
            os.environ["LOCOHD_NO_TILES"] = "1"
        for n, outs in ((20_000, ("device", "host")), (50_000, ("device",))):
            name = f"condensed_{n}_{route}"
            if args.only not in name:
                continue
            for where in outs:
                if where == "device":
                    vec = torch.empty(n * (n - 1) // 2, dtype=torch.float64, device="cuda")
                    mat = torch.empty((n, n), dtype=torch.float64, device="cuda")
                    kv, km = dict(out=vec.data_ptr()), dict(scores=mat.data_ptr())
                else:
                    kv, km = {}, {}
                t0 = ctx.tile_launches
                alternated(f"{name}_{where}",
                           ("condensed", n * (n - 1) // 2, lambda: ctx.score_condensed(env, 0, n, **kv)),
                           ("matrix", n * n, lambda: ctx.score_cross(env, env, 0, n, 0, n, **km)))
                emit({"name": f"{name}_{where}_tile_launches", "tile_launches": ctx.tile_launches - t0})
                if where == "device":
                    iu = torch.triu_indices(n, n, 1, device="cuda")
                    upper = mat[iu[0], iu[1]]
                    del iu
                    same = bool(torch.equal(upper.view(torch.int64), vec.view(torch.int64)))
                    emit({"name": f"{name}_device_equals_matrix_upper_triangle", "bit_identical": same})
                    del upper, vec, mat
                    torch.cuda.empty_cache()
    os.environ.pop("LOCOHD_NO_TILES", None)


main()
