"""A/B of the triangulation node kernel on hypersim100 (the bench workload, one pipeline group): the split form
(tri_gen_kernel + tri_score_kernel) against the fused tri_node_kernel (LIMAP_B200_TRI_FUSED=1), alternating in one
process. Prints one JSON line: median / min / max node-kernel time and run time of both, with the card's name, power
limit and SM clock.
  python scripts/tri_split_ab.py [runs per arm, default 20]"""
import json
import os
import subprocess
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        return dict(zip(q.split(","), [x.strip() for x in out.split(",")]))
    except (OSError, subprocess.SubprocessError):
        return {}


def main():
    from limap_b200.config import DEFAULT_YAML_TRIANGULATION
    from limap_b200.engine import TriEngine
    from limap_b200.synth import CONFIGS, make_scene
    n = int(sys.argv[1]) if len(sys.argv) > 1 else 20
    sc = make_scene(**CONFIGS["hypersim100"])
    eng = TriEngine(dict(DEFAULT_YAML_TRIANGULATION))
    eng.upload(sc)
    eng.set_ranges(*sc.ranges)
    eng.add_matches_bulk(*sc.bulk_matches())
    eng.set_pipeline_groups(1)
    arms = {"fused": "1", "split": None}
    res = {k: {"kernel_ms": [], "run_ms": []} for k in arms}
    for it in range(n + 2):  # two warm-up rounds
        for k, v in arms.items():
            if v is None:
                os.environ.pop("LIMAP_B200_TRI_FUSED", None)
            else:
                os.environ["LIMAP_B200_TRI_FUSED"] = v
            st = eng.run()
            if it >= 2:
                res[k]["kernel_ms"].append(st["last_node_kernel_ms"])
                res[k]["run_ms"].append(st["last_run_ms"])
    os.environ.pop("LIMAP_B200_TRI_FUSED", None)
    out = {"workload": "hypersim100", "runs_per_arm": n, "gpu": gpu_info(), "n_candidates": int(st["n_candidates"])}
    for k, r in res.items():
        for m, xs in r.items():
            xs = np.asarray(xs)
            out[f"{k}_{m}"] = {"median": float(np.median(xs)), "min": float(xs.min()), "max": float(xs.max()),
                               "iqr": float(np.percentile(xs, 75) - np.percentile(xs, 25))}
    out["kernel_speedup"] = out["fused_kernel_ms"]["median"] / out["split_kernel_ms"]["median"]
    print(json.dumps(out))


if __name__ == "__main__":
    main()
