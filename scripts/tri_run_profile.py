"""Kernel table of one warmed-up triangulation run on hypersim100 (the bench workload), from torch.profiler with CUDA
activities. Writes OUTDIR/tri_run_profile.txt (and prints it): the card's name, power limit and SM clock, then every
kernel and copy of the run with its count and summed device time, the row-preparation kernels (match rows -> node-major
rows and node offsets) summed separately, and the span from the first kernel start to the last kernel end.
  python scripts/tri_run_profile.py OUTDIR [--groups G] [--row-sort cub]"""
import argparse
import os
import re
import subprocess
import sys
from collections import OrderedDict

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

# kernels that turn the uploaded match tables into node-major rows and node row offsets
PREP = ("expand_rows_kernel", "expand_exhaustive_kernel", "DeviceRadixSortHistogramKernel",
        "DeviceRadixSortExclusiveSumKernel", "DeviceRadixSortOnesweepKernel", "node_offsets_kernel",
        "row_views_kernel", "row_count_kernel", "row_scan_kernel", "row_scatter_kernel")


def gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        return dict(zip(q.split(","), [x.strip() for x in out.split(",")]))
    except (OSError, subprocess.SubprocessError):
        return {}


def short_name(name):
    """'void lm::foo_kernel<true>(lm::TriParams)' -> 'foo_kernel<true>'; CUB kernels keep their class name only."""
    base = name.split("(")[0].replace("void ", "").strip()
    m = re.match(r"^([\w:]+)(<.*>)?$", base)
    if not m:
        return base[:80]
    ident = m.group(1).split("::")[-1]
    targs = m.group(2) or ""
    if ident.startswith("DeviceRadixSort") or ident.startswith("Device") or len(targs) > 24:
        return ident
    return ident + targs


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("outdir")
    ap.add_argument("--groups", type=int, default=1)
    ap.add_argument("--row-sort", default=None, help="value of LIMAP_B200_ROW_SORT for the run (e.g. cub)")
    a = ap.parse_args()
    import torch
    from torch.profiler import ProfilerActivity, profile

    from limap_b200.config import DEFAULT_YAML_TRIANGULATION
    from limap_b200.engine import TriEngine
    from limap_b200.synth import CONFIGS, make_scene
    if a.row_sort:
        os.environ["LIMAP_B200_ROW_SORT"] = a.row_sort
    info = gpu_info()
    sc = make_scene(**CONFIGS["hypersim100"])
    eng = TriEngine(dict(DEFAULT_YAML_TRIANGULATION))
    eng.upload(sc)
    eng.set_ranges(*sc.ranges)
    eng.add_matches_bulk(*sc.bulk_matches())
    eng.set_pipeline_groups(a.groups)
    for _ in range(3):
        eng.run()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        st = eng.run()
        torch.cuda.synchronize()
    info_after = gpu_info()
    rows = OrderedDict()
    t0, t1 = None, None
    for e in prof.events():
        if e.device_type != torch.autograd.DeviceType.CUDA:
            continue
        k = short_name(e.name)
        us = e.time_range.elapsed_us()
        t0 = e.time_range.start if t0 is None else min(t0, e.time_range.start)
        t1 = e.time_range.end if t1 is None else max(t1, e.time_range.end)
        n, tot = rows.get(k, (0, 0.0))
        rows[k] = (n + 1, tot + us)
    lines = [f"hypersim100, {a.groups} pipeline group(s), LIMAP_B200_ROW_SORT={a.row_sort or '(default)'}",
             f"gpu before: {info}", f"gpu after:  {info_after}",
             f"run stats: last_run_ms {st['last_run_ms']:.4f}  last_node_kernel_ms {st['last_node_kernel_ms']:.4f}  "
             f"n_rows {int(st['n_rows'])}",
             f"{'kernel / copy':<48}{'count':>6}{'total us':>12}{'mean us':>10}"]
    prep = 0.0
    for k, (n, tot) in sorted(rows.items(), key=lambda kv: -kv[1][1]):
        lines.append(f"{k:<48}{n:>6}{tot:>12.1f}{tot / n:>10.1f}")
        if any(k.startswith(p) for p in PREP):
            prep += tot
    lines.append(f"row preparation kernels (expand / sort / node offsets, or count / scan / scatter): {prep:.1f} us")
    if t0 is not None:
        lines.append(f"first kernel start -> last kernel end: {t1 - t0:.1f} us")
    text = "\n".join(lines)
    print(text)
    os.makedirs(a.outdir, exist_ok=True)
    suffix = f"_g{a.groups}" + (f"_{a.row_sort}" if a.row_sort else "")
    with open(os.path.join(a.outdir, f"tri_run_profile{suffix}.txt"), "w") as f:
        f.write(text + "\n")


if __name__ == "__main__":
    main()
