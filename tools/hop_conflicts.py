"""Shared-memory bank conflicts of the TAG layer kernels' hop gathers and level stores under both swizzle-key policies (CPU only).

Builds each grid's batch the way dss2_graph_build tiles it (host model in dss2.graph), assigns the keys with the library's own host
routine, and counts the wavefronts of every 8-row access phase against the conflict-free count (dss2.graph.hop_wavefronts).  The
large-graph configurations (a graph above 256 buses) run without tiles and are not listed.

    python tools/hop_conflicts.py [--batch 4096]
"""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "deep-statistical-solver-for-distribution-system-state-estimation_b200"))

from dss2 import graph, synth  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=4096)
    ap.add_argument("--tile-cap", type=int, default=256)
    args = ap.parse_args()
    rows = []
    for case in ("ober_sub", "cigre14", "cigre14_reswitched"):
        st = synth.synthetic_store(synth.load_grid(case), 1, device="cpu")
        ei, n = st.edge_index.numpy(), st.max_nodes
        ci, tp = graph.host_ell(np.concatenate([ei + b * n for b in range(args.batch)], axis=1), np.arange(args.batch + 1) * n, args.tile_cap)
        for policy in ("identity", "color"):
            w = graph.hop_wavefronts(ci, tp, graph.host_hop_keys(ci, tp, policy))
            rows.append({"grid": case, "batch": args.batch, "tiles": len(tp) - 1, "policy": policy,
                         "gather_wavefronts": w["gather"][0], "gather_ideal": w["gather"][1], "gather_ratio": round(w["gather"][0] / w["gather"][1], 3),
                         "store_wavefronts": w["store"][0], "store_ideal": w["store"][1], "store_ratio": round(w["store"][0] / w["store"][1], 3)})
            print(json.dumps(rows[-1]))


if __name__ == "__main__":
    main()
