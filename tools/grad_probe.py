"""Cost of the coordinate gradients: median time per call of from_primitives against from_primitives_grad on the
configuration-1 shape (450 primitives, 150 anchors) and the configuration-2 shape (10 000 primitives, 10 000
anchors), through the C ABI and through LoCoHD.from_arrays / from_arrays_grad.  Host inputs and outputs; every call
ends in a device synchronisation.  Prints one JSON line per shape and writes them to --out when given."""
import argparse
import json
import subprocess
import sys
import time
from pathlib import Path

import numpy as np

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
from benchdata import synth  # noqa: E402
from loco_hd_b200 import _capi  # noqa: E402


def median_ms(f, warmup, reps):
    for _ in range(warmup):
        f()
    times = []
    for _ in range(reps):
        t0 = time.perf_counter()
        f()
        times.append(time.perf_counter() - t0)
    return 1e3 * float(np.median(times))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import loco_hd

    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    ctx = _capi.Context(0)
    rows = []
    for key, (a, b), step in (("cfg1_150_anchors", synth.config1(), None),
                              ("cfg2_10000_anchors", synth.config2_pair(0), 1)):
        wf = ("uniform", (3.0, 10.0)) if step is None else ("kumaraswamy", (3.0, 10.0, 2.0, 5.0))
        step = a.k if step is None else step
        anchors = np.stack([np.arange(0, a.n, step, dtype=np.uint32)] * 2, axis=1)
        ctx.set_params(7, [wf], tag_rule={"accept_same": False})
        lchd = loco_hd.LoCoHD([f"T{i}" for i in range(7)], loco_hd.WeightFunction(wf[0], list(wf[1])),
                              loco_hd.TagPairingRule({"accept_same": False}))
        A, B = (a.xyz, a.cat, a.tag), (b.xyz, b.cat, b.tag)
        calls = {"c_abi": lambda: ctx.from_primitives(*A, *B, anchors, 10.0),
                 "c_abi_grad": lambda: ctx.from_primitives_grad(*A, *B, anchors, 10.0),
                 "from_arrays": lambda: lchd.from_arrays(*A, *B, anchors, 10.0),
                 "from_arrays_grad": lambda: lchd.from_arrays_grad(*A, *B, anchors, 10.0)}
        row = {"shape": key, "anchor_pairs": len(anchors), "gpu": gpu, "reps": args.reps}
        for name, f in calls.items():
            row[name + "_ms"] = median_ms(f, args.warmup, args.reps)
        row["grad_over_score_c_abi"] = row["c_abi_grad_ms"] / row["c_abi_ms"]
        row["grad_over_score_from_arrays"] = row["from_arrays_grad_ms"] / row["from_arrays_ms"]
        print(json.dumps(row), flush=True)
        rows.append(row)
    ctx.close()
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text("".join(json.dumps(r) + "\n" for r in rows))


if __name__ == "__main__":
    main()
