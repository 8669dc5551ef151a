"""A/B of the swizzle-key policies (DSS2_HOP_KEYS = identity | color) on the flagship workload, in one process tree on one GPU.

First one bench.py run per policy with --dump-outputs: the dumped outputs and the loss-trajectory hash must be byte-identical (the keys
move bytes only).  Then --pairs alternating pairs of bench.py runs (identity first in even pairs, color first in odd ones), each
reporting ms_per_step and the per-launch times of the TAG layer kernels from its roofline section.  The card's name, power limit and
clocks are read in the same call.  Writes --out (default profiles/r3d_hop_keys.json).

    python tools/hop_keys_ab.py --pairs 5 --steps 50 --warmup 5
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def card():
    q = "name,power.limit,clocks.max.sm,clocks.sm"
    r = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True)
    first = r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else ""
    return dict(zip(q.split(","), (v.strip() for v in first.split(",")))) if first else {"error": r.stderr.strip()}


def bench(policy, args, dump=None):
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(args.steps), "--warmup", str(args.warmup),
           "--no-cpu-baseline", "--no-e2e"]
    if dump:
        cmd += ["--dump-outputs", dump]
    run = subprocess.run(cmd, capture_output=True, text=True, cwd=tempfile.gettempdir(), env={**os.environ, "DSS2_HOP_KEYS": policy})
    if run.returncode != 0:
        sys.exit(f"bench.py ({policy}) failed:\n{run.stderr[-3000:]}")
    res = json.loads(run.stdout.strip().splitlines()[-1])
    kern = {r["kernel"].split(" ")[0]: r["us_per_launch"] for r in (res.get("roofline") or {}).get("all_layer_kernels", [])}
    return {"ms_per_step": res["ms_per_step"], "sha": res.get("loss_trajectory_sha256_16"), "kernels_us": kern, "clocks": res.get("clocks")}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--pairs", type=int, default=5)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r3d_hop_keys.json"))
    args = ap.parse_args()
    out = {"card_before": card(), "workload": "bench.py --gpus 1 (SkipPFN train step, Oberrhein B=4096), --no-e2e --no-cpu-baseline",
           "steps": args.steps, "warmup": args.warmup}
    # bit-identity first
    with tempfile.TemporaryDirectory() as tmp:
        first = {}
        for policy in ("identity", "color"):
            first[policy] = bench(policy, args, dump=os.path.join(tmp, policy))
        names = sorted(os.listdir(os.path.join(tmp, "identity")))
        same = names == sorted(os.listdir(os.path.join(tmp, "color"))) and all(
            np.load(os.path.join(tmp, "identity", n)).tobytes() == np.load(os.path.join(tmp, "color", n)).tobytes() for n in names)
    out["bit_identical"] = {"dump_outputs": same, "dumped_arrays": len(names), "loss_trajectory_sha256_16": {p: r["sha"] for p, r in first.items()},
                            "sha_equal": first["identity"]["sha"] == first["color"]["sha"]}
    print(json.dumps(out["bit_identical"]), flush=True)
    if not (same and out["bit_identical"]["sha_equal"]):
        sys.exit("outputs differ between the key policies")
    runs = {"identity": [], "color": []}
    for i in range(args.pairs):
        for policy in (("identity", "color") if i % 2 == 0 else ("color", "identity")):
            r = bench(policy, args)
            runs[policy].append(r)
            print(policy, round(r["ms_per_step"], 4), {k: round(v, 2) for k, v in r["kernels_us"].items() if k.startswith("k_tag")}, flush=True)
    summ = {}
    for policy, rs in runs.items():
        ms = [r["ms_per_step"] for r in rs]
        kern = {k: statistics.median(r["kernels_us"][k] for r in rs) for k in rs[0]["kernels_us"]}
        summ[policy] = {"ms_per_step": ms, "median": statistics.median(ms), "min": min(ms), "max": max(ms), "kernels_us_median": kern,
                        "clocks": [r["clocks"] for r in rs]}
    ratio = [c["ms_per_step"] / i["ms_per_step"] for i, c in zip(runs["identity"], runs["color"])]
    out.update(runs=summ, color_over_identity_per_pair=ratio, color_over_identity_median=statistics.median(ratio), card_after=card())
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps({p: {k: v for k, v in s.items() if k != "clocks"} for p, s in summ.items()}, indent=1))
    print("color / identity per pair:", [round(r, 4) for r in ratio], "median", round(statistics.median(ratio), 4))


if __name__ == "__main__":
    main()
