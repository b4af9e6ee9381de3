"""A/B of the row preparation on hypersim100 (the bench workload, one pipeline group by default): the per-view counting
sort (row_count / row_scan / row_scatter, the default) against the radix-sort path (LIMAP_B200_ROW_SORT=cub),
alternating in one process on one engine. Prints one JSON line: median / min / max / IQR of the run time and of the
node-kernel time of both, with the card's name, power limit and SM clock.
  python scripts/row_sort_ab.py [runs per arm, default 20] [pipeline groups, default 1]"""
import json
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from scripts.tri_split_ab import gpu_info  # noqa: E402


def main():
    from limap_b200.config import DEFAULT_YAML_TRIANGULATION
    from limap_b200.engine import TriEngine
    from limap_b200.synth import CONFIGS, make_scene
    n = int(sys.argv[1]) if len(sys.argv) > 1 else 20
    groups = int(sys.argv[2]) if len(sys.argv) > 2 else 1
    sc = make_scene(**CONFIGS["hypersim100"])
    eng = TriEngine(dict(DEFAULT_YAML_TRIANGULATION))
    eng.upload(sc)
    eng.set_ranges(*sc.ranges)
    eng.add_matches_bulk(*sc.bulk_matches())
    eng.set_pipeline_groups(groups)
    arms = {"cub": "cub", "counting": None}
    res = {k: {"run_ms": [], "kernel_ms": []} for k in arms}
    info = gpu_info()
    for it in range(n + 2):  # two warm-up rounds
        for k, v in arms.items():
            if v is None:
                os.environ.pop("LIMAP_B200_ROW_SORT", None)
            else:
                os.environ["LIMAP_B200_ROW_SORT"] = v
            st = eng.run()
            if it >= 2:
                res[k]["run_ms"].append(st["last_run_ms"])
                res[k]["kernel_ms"].append(st["last_node_kernel_ms"])
    os.environ.pop("LIMAP_B200_ROW_SORT", None)
    out = {"workload": "hypersim100", "pipeline_groups": groups, "runs_per_arm": n, "gpu": info,
           "gpu_after": gpu_info(), "n_candidates": int(st["n_candidates"])}
    for k, r in res.items():
        for m, xs in r.items():
            xs = np.asarray(xs)
            out[f"{k}_{m}"] = {"median": float(np.median(xs)), "min": float(xs.min()), "max": float(xs.max()),
                               "iqr": float(np.percentile(xs, 75) - np.percentile(xs, 25))}
    out["run_ms_saved"] = out["cub_run_ms"]["median"] - out["counting_run_ms"]["median"]
    print(json.dumps(out))


if __name__ == "__main__":
    main()
