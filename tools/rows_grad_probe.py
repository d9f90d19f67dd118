"""Cost of the gradients of from_coords and from_dmxs: from_coords against from_coords_grad and from_dmxs against
from_dmxs_grad through the C ABI, at n = 1000, 2000 and 5000 points (C = 7, uniform [3, 10], Hellinger-2; random
clouds at protein-like density, B = A moved by 0.5 A).  Host inputs and outputs, as a caller of the reference API has
them.  Per call, after a warm-up, the median of
  * wall_ms:   host clock around the call, which ends in a device synchronisation (uploads and downloads included);
  * device_ms: the library's own CUDA events around its kernel groups (Context.profile_read), summed over the call.
The plain from_coords / from_dmxs is the two row sets (envset_from_coords / envset_from_rows) plus score_pairs, the
calls LoCoHD.from_coords / from_dmxs make.  Prints one JSON line per size, with the card's name and power limit read
in the same run, and writes them to --out when given."""
import argparse
import json
import subprocess
import sys
import time
from pathlib import Path

import numpy as np

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
sys.path.insert(0, str(Path(__file__).resolve().parent.parent / "tests"))
from loco_hd_b200 import _capi  # noqa: E402
from rows_grad_reference import euclidean_rows  # noqa: E402


def measure(ctx, f, warmup, reps):
    for _ in range(warmup):
        f()
    ctx.profile_enable(True)
    ctx.profile_read()
    wall, dev = [], []
    for _ in range(reps):
        t0 = time.perf_counter()
        f()
        wall.append(time.perf_counter() - t0)
        dev.append(sum(ms for ms, _ in ctx.profile_read().values()))
    ctx.profile_enable(False)
    return 1e3 * float(np.median(wall)), float(np.median(dev))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="1000,2000,5000")
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()[0]
    ctx = _capi.Context(0)
    ctx.set_params(7, [("uniform", (3.0, 10.0))])
    rows = []
    for n in (int(v) for v in args.sizes.split(",")):
        rng = np.random.default_rng(n)
        side = (n / 0.01) ** (1 / 3)   # ~0.01 points per cubic Angstrom
        xa = rng.uniform(0, side, (n, 3))
        xb = xa + rng.normal(0, 0.5, (n, 3))
        ca = rng.integers(0, 7, n).astype(np.uint16)
        cb = ca.copy()
        cb[rng.integers(0, n, n // 10)] = rng.integers(0, 7, n // 10)
        ta, tb = euclidean_rows(xa), euclidean_rows(xb)
        pairs = np.stack([np.arange(n)] * 2, axis=1).astype(np.uint32)

        def plain(build_a, build_b):
            ea, eb = build_a(), build_b()
            s = ctx.score_pairs(ea, eb, pairs)
            ea.close(); eb.close()
            return s
        calls = {"from_coords": lambda: plain(lambda: ctx.envset_from_coords(xa, ca), lambda: ctx.envset_from_coords(xb, cb)),
                 "from_coords_grad": lambda: ctx.from_coords_grad(xa, ca, xb, cb),
                 "from_dmxs": lambda: plain(lambda: ctx.envset_from_rows(ta, ca), lambda: ctx.envset_from_rows(tb, cb)),
                 "from_dmxs_grad": lambda: ctx.from_rows_grad(ta, ca, tb, cb)}
        s_coords, s_grad = calls["from_coords"](), calls["from_coords_grad"]()[0]
        row = {"n_points": n, "categories": 7, "weight_function": "uniform [3, 10]", "statistical_distance": "Hellinger-2",
               "gpu_name_power_limit": gpu, "reps": args.reps, "warmup": args.warmup,
               "max_abs_score_diff_grad_vs_plain": float(np.abs(s_coords - s_grad).max())}
        for name, f in calls.items():
            row[name + "_wall_ms"], row[name + "_device_ms"] = measure(ctx, f, args.warmup, args.reps)
        row["coords_grad_over_plain_wall"] = row["from_coords_grad_wall_ms"] / row["from_coords_wall_ms"]
        row["dmxs_grad_over_plain_wall"] = row["from_dmxs_grad_wall_ms"] / row["from_dmxs_wall_ms"]
        print(json.dumps(row), flush=True)
        rows.append(row)
    ctx.close()
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text("".join(json.dumps(r) + "\n" for r in rows))


if __name__ == "__main__":
    main()
