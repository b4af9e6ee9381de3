#!/usr/bin/env python
"""bench.py — headline benchmark of the line-triangulation hot path (BASELINE.json metric
"3D line candidates triangulated+scored/sec").

A step = one pass of candidate generation + scoring + selection (all TriangulateImage calls of a scene,
SURVEY.md §8d M1) over one synthetic scene of BASELINE.json configs[1] shape ("hypersim100": V=100 views,
L=1000 lines/view, N=20 neighbours, K=10 matches per line per neighbour = 2e7 match rows). The unit
counted is the match row tested by triangulateOneNode.

  value : whole-job rows/s with the scene and match tables already resident in HBM (CUDA-event timed,
          max over ranks).
  e2e   : the same metric through the public engine API with HOST (pinned) buffers: scene upload,
          match upload, run (+ the multi-GPU exchange), per-node results + valid connections read back, every step.
  roofline : the fused generate+score kernel against the measured HBM copy bandwidth
          (MEASURED_PEAKS.json), algorithmic bytes per SURVEY.md §8(d); `compute` = pipe utilisation of the same
          kernel from the committed ncu capture (profiles/r02_kernel_metrics.json).
  cpu_baseline : CPU implementations of the same path on this host's cores. One rule on every box: `value` is the
          fp64 restatement (oracle/, "port") with the OpenMP loop moved out to the 2D lines of an image (identical
          results) on ALL usable cores -- the best CPU number; `reference_schedule` is the reference's own sources
          compiled unchanged (oracle/_ref, `kind: "reference"`; the restatement with the reference's loop structure if
          that library is missing) with the reference's OpenMP schedule at its fastest thread count.
  parity : the CPU leg's results are compared with the timed GPU run's (candidate counts, best candidate ids, valid
          connections bit-exact; endpoints 1e-4) instead of being thrown away.

N > 1 (torchrun): equal-work weak scaling. The scene is N independent blocks of the hypersim100 shape (block b =
seed 1235 + 1000 b; block 0 is the N=1 scene), 100 N views in ONE replicated scene; rank r triangulates block r
(sharding by source image, SURVEY.md §8e) and the per-node results of all ranks are exchanged with ONE NCCL
all-gather inside the timed region (pack kernel -> all_gather_into_tensor -> unpack kernel, no host sync).

Other legs on the same line: `lm_ba` (configs[3], M2), `remerge` (§8f-1), `jlinkage` (a18, configs[4] slice),
`sweep500` (configs[2], strong scaling of one fixed scene).

--impl reference times the reference's own compiled sources (oracle/_ref; the restatement if missing) on bounded
samples of the same scene and prints the best-CPU port beside it.

--dump-outputs DIR writes what the timed path computed in its last step (dump_outputs) as DIR/<name>.npy; the scene is
seeded, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "3D line candidates triangulated+scored/sec"
UNIT = "match rows/s"
WORKLOAD = "hypersim100"
FP64_NOMINAL_TFLOPS = 40.0  # SURVEY.md §8(d) nominal non-tensor fp64 peak of B200


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def load_kernel_metrics():
    """ncu-derived per-kernel figures of the committed build (profiles/r02_kernel_metrics.json): DRAM traffic per
    launch and pipe utilisation. Never measured under bench.py itself."""
    try:
        with open(os.path.join(ROOT, "profiles", "r02_kernel_metrics.json")) as f:
            return json.load(f)
    except (OSError, ValueError):
        return {}


class ClockSampler:
    """Samples nvidia-smi SM clocks / throttle reasons while the timed region runs."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index=0):
        self.gpu = gpu_index
        self.rows = []
        self._stop = threading.Event()
        self._t = None

    def _run(self):
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                      "-i", str(self.gpu)], capture_output=True, text=True, timeout=5).stdout
                for line in out.strip().splitlines():
                    self.rows.append([x.strip() for x in line.split(",")])
            except Exception:
                pass
            self._stop.wait(0.1)

    def start(self):
        self._t = threading.Thread(target=self._run, daemon=True)
        self._t.start()

    def stop(self):
        self._stop.set()
        if self._t:
            self._t.join(timeout=6)
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[1]))
                mx.append(float(r[2]))
                for k, n in enumerate(names):
                    if r[5 + k].lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                continue
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons),
                "samples": len(sm)}


def get_scene(n_gpus, rank):
    """N=1: the hypersim100 scene. N>1: N blocks of that shape in one scene, matches only for this rank's block."""
    from limap_b200.synth import CONFIGS, concat_scenes, make_scene
    cfg = dict(CONFIGS[WORKLOAD])
    per = cfg["V"]
    if n_gpus == 1:
        return make_scene(**cfg), per
    blocks = []
    for b in range(n_gpus):
        c = dict(cfg)
        c["seed"] = cfg["seed"] + 1000 * b
        blocks.append(make_scene(match_views=None if b == rank else [], **c))
    return concat_scenes(blocks), per


def algorithmic_bytes(n_rows, n_nodes, n_views, n_cand, n_valid):
    """SURVEY.md §8(d): B_gen + B_score for the fused kernel (fp32-storage convention of the survey)."""
    b_gen = 24 * n_rows + 16 * n_nodes + 44 * n_views + 48 * n_cand
    b_score = n_cand * (48 + 16) + 4 * n_cand + n_nodes * 48 + 4 * n_valid
    return b_gen + b_score


def reference_impl():
    """(constructor, kind): the reference's own compiled sources (oracle/_ref, built by build() where the reference's
    sources are present and shipped as object code) when they load here, else the restatement with the reference's loop
    structure."""
    from oracle import oracle as orc
    try:
        from oracle import ref
        if ref.available():
            ref.lib()
            return (lambda cfg, threads: ref.RefTri(cfg, threads=threads)), "reference"
    except Exception:
        pass
    return (lambda cfg, threads: orc.OracleTri(cfg, threads=threads)), "port"


def pick_cpu_threads(scene, make=None):
    """The reference parallelises with OpenMP inside one node (n ~ 10..200 iterations per region), which does
    not scale to every core of a large host; calibrate on one source image and keep the fastest count."""
    from limap_b200.config import DEFAULT_YAML_TRIANGULATION
    from oracle import oracle as orc
    if make is None:
        make = reference_impl()[0]
    n = orc.usable_cpus()
    cands = sorted({1, min(8, n), min(32, n), n})
    i0 = sorted(scene.matches)[0]
    f = scene.flat_matches(i0)
    best, best_t = 1, None
    for th in cands:
        o = make(dict(DEFAULT_YAML_TRIANGULATION), th)
        o.upload(scene)
        o.set_ranges(*scene.ranges)
        t0 = time.perf_counter()
        o.add_image_matches(i0, *f)
        dt = time.perf_counter() - t0
        if best_t is None or dt < best_t:
            best, best_t = th, dt
        del o
    return best


def tri_parity(eng, o, img_ids, tol=1e-4):
    """GPU engine vs oracle on the given source images: candidate counts, best-candidate ids and valid connections
    bit-exact, endpoints/depths/uncertainty within `tol`, scores within 1e-6."""
    rows = nodes = bad_count = bad_best = bad_edges = 0
    worst = 0.0
    for i in img_ids:
        gl, gng, gnc = eng.get_best(i)
        ol, ong, onc = o.get_best(i)
        nodes += len(onc)
        bad_count += int((gnc != onc).sum())
        has = (onc > 0) & (gnc == onc)
        bad_best += int((gng[has] != ong[has]).any(axis=1).sum())
        if has.any():
            worst = max(worst, float(np.abs(gl[has, :9] - ol[has, :9]).max()))
            bad_best += int((np.abs(gl[has, 9] - ol[has, 9]) > 1e-6).sum())
        goff, ge = eng.get_valid_edges(i)
        ooff, oe = o.get_valid_edges(i)
        if not np.array_equal(goff, ooff):
            bad_edges += int((np.diff(goff) != np.diff(ooff)).sum())
        else:
            node_of = np.repeat(np.arange(len(goff) - 1), np.diff(goff))
            ga = np.stack([node_of, ge[:, 0], ge[:, 1]], 1) if len(ge) else np.zeros((0, 3), np.int64)
            oa = np.stack([node_of, oe[:, 0], oe[:, 1]], 1) if len(oe) else np.zeros((0, 3), np.int64)
            ga = ga[np.lexsort((ga[:, 2], ga[:, 1], ga[:, 0]))]
            oa = oa[np.lexsort((oa[:, 2], oa[:, 1], oa[:, 0]))]
            bad_edges += int((ga != oa).any(axis=1).sum())
    return {"images": len(img_ids), "nodes": int(nodes), "count_mismatches": bad_count, "best_mismatches": bad_best,
            "valid_edge_mismatches": bad_edges, "max_abs_endpoint_diff": worst,
            "ok": bool(bad_count == 0 and bad_best == 0 and bad_edges == 0 and worst <= tol)}


def run_reference(args, rank, world):
    """Reference arm: the reference's own CPU implementation of the path on this host's cores -- its hot-path sources
    compiled unchanged (oracle/_ref, `kind: "reference"`; Eigen / COLMAP headers replaced by oracle/ref_shim, object
    code shipped with the repo snapshot) with the reference's own OpenMP schedule at its fastest thread count; the
    restatement (`kind: "port"`) only if that library does not load. Every step is a bounded sample of hypersim100.
    `best_cpu_port` on the same line: the restatement with the OpenMP loop moved out to the 2D lines of an image
    (identical results, all cores) -- what a throughput-tuned CPU implementation reaches on this box."""
    if rank != 0:
        return
    from limap_b200.config import DEFAULT_YAML_TRIANGULATION
    from oracle import oracle as orc
    orc.build()
    scene, per = get_scene(1, 0)
    make, kind = reference_impl()
    cores = pick_cpu_threads(scene, make)
    ids = [int(i) for i in scene.img_ids]
    flat = {i: scene.flat_matches(i) for i in ids}
    nsteps = args.warmup + args.steps

    def mk():
        o = make(dict(DEFAULT_YAML_TRIANGULATION), cores)
        o.upload(scene)
        o.set_ranges(*scene.ranges)
        return o

    sample_imgs = args.ref_images
    if sample_imgs <= 0:  # size the sample so that the whole arm takes about args.ref_seconds
        o = mk()
        t0 = time.perf_counter()
        o.add_image_matches(ids[0], *flat[ids[0]])
        t_img = time.perf_counter() - t0
        del o
        sample_imgs = int(min(len(ids), max(3, args.ref_seconds / (max(nsteps, 1) * t_img))))
    times, rows = [], []
    for s in range(nsteps):
        o = mk()
        pick = [ids[(s * sample_imgs + k) % len(ids)] for k in range(sample_imgs)]
        t0 = time.perf_counter()
        for i in pick:
            o.add_image_matches(i, *flat[i])
        dt = time.perf_counter() - t0
        if s >= args.warmup:
            times.append(dt)
            rows.append(o.rows_tested())
        del o
    value = float(sum(rows) / sum(times))
    what = ("the reference's own sources (oracle/_ref)" if kind == "reference" else "oracle port, reference loop structure")
    sample = (f"{sample_imgs} of the {len(ids)} source images per step ({int(np.mean(rows))} rows), {args.steps} steps; "
              f"{what}, OpenMP threads = {cores} (fastest of 1/8/32/all on this host)")
    best = None
    try:  # the throughput-tuned schedule, for the record
        o = orc.OracleTri(dict(DEFAULT_YAML_TRIANGULATION), threads=orc.usable_cpus(), node_parallel=True)
        o.upload(scene)
        o.set_ranges(*scene.ranges)
        t0 = time.perf_counter()
        for i in ids[:max(5, min(len(ids), 3 * sample_imgs))]:
            o.add_image_matches(i, *flat[i])
            if time.perf_counter() - t0 > 10.0:
                break
        best = {"value": o.rows_tested() / (time.perf_counter() - t0), "unit": UNIT, "cores": orc.usable_cpus(),
                "kind": "port", "schedule": "OpenMP over the 2D lines of an image (identical results)"}
    except Exception as e:
        best = {"error": str(e)}
    line = {"metric": METRIC, "value": value, "unit": UNIT, "impl": "reference", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * float(np.mean(times)),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic",
            "config": {"workload": WORKLOAD, "V": 100, "L": 1000, "N": 20, "K": 10, "sample": sample},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample,
                             "host_cpus": orc.usable_cpus()},
            "best_cpu_port": best,
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


DUMP_BUDGET_BYTES = 64 << 20


def dump_outputs(eng, out_dir, node_begin, node_end):
    """What a caller of TriEngine.run() receives for the nodes [node_begin, node_end) (this rank's own source images),
    as float64 .npy files: each node's record (best candidate's 3D line = start, end, two depths, uncertainty; its
    score; its neighbour (image id, line id); candidate and valid-connection counts) and its valid connections (neighbour
    image id, line id), sorted within each node because they form a set. `node_index` holds the scene-wide index of each
    dumped node: all of them, or a fixed seeded sample of them when the whole would exceed DUMP_BUDGET_BYTES."""
    nodes = eng.get_nodes()
    off, edges = eng.get_all_valid_edges()
    idx = np.arange(node_begin, node_end)
    n_edges = int(off[node_end] - off[node_begin])
    per_node, per_edge = 8 * 16, 8 * 2  # bytes per node (15 values, its index, its offset), per valid connection
    total = per_node * len(idx) + per_edge * n_edges
    if total > DUMP_BUDGET_BYTES:
        k = int(0.9 * len(idx) * DUMP_BUDGET_BYTES / total)  # 10% margin: connection counts vary from node to node
        idx = np.sort(np.random.default_rng(0).choice(idx, k, replace=False))
    cnt = off[idx + 1] - off[idx]
    starts = np.concatenate([[0], np.cumsum(cnt)])
    rows = np.repeat(off[idx] - starts[:-1], cnt) + np.arange(int(starts[-1]))
    node_of = np.repeat(np.arange(len(idx)), cnt)
    e = edges[rows]
    e = e[np.lexsort((e[:, 1], e[:, 0], node_of))]
    nodes = nodes[idx]
    arrays = {"node_index": idx, "node_line": nodes["line"], "node_score": nodes["score"],
              "node_best_neighbor": np.stack([nodes["ng_view"], nodes["ng_line"]], 1),
              "node_counts": np.stack([nodes["n_cand"], nodes["n_valid"]], 1),
              "valid_edge_off": starts, "valid_edges": e}
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a, np.float64))


def bind_to_gpu_numa_node(local_rank):
    """One process per GPU: run on (and therefore allocate pinned host buffers from) the CPU cores next to this rank's
    GPU, so that N ranks uploading at once do not pull their pages across the socket interconnect. Best effort."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(local_rank)
        n_words = (os.cpu_count() + 63) // 64
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, n_words)
        cpus = {64 * w + b for w, m in enumerate(mask) for b in range(64) if (int(m) >> b) & 1}
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            return len(cpus)
    except Exception:
        pass
    return None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--ref-images", type=int, default=0, help="source images per reference step (0: sized from --ref-seconds)")
    ap.add_argument("--ref-seconds", type=float, default=90.0, help="time budget of the whole --impl reference arm")
    ap.add_argument("--cpu-seconds", type=float, default=16.0, help="budget of the cpu_baseline legs")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-lm", action="store_true", help="skip the lm_ba / remerge / jlinkage / sweep500 legs")
    ap.add_argument("--groups", type=int, default=8, help="pipeline groups of the e2e path (upload/run overlap)")
    ap.add_argument("--value-groups", type=int, default=1,
                    help="pipeline groups of the device-resident leg (1: the node kernel runs alone and is timed cleanly for the "
                         "roofline; >1 hides the row preparation of group g+1 under the node kernel of group g)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the outputs of the last timed step for rank 0's source images as DIR/<name>.npy")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3) if args.impl == "native" else args.warmup
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    # stdout carries exactly ONE line (the JSON): everything native libraries print (NCCL's version banner goes to fd 1
    # whatever NCCL_DEBUG_FILE says) is redirected to stderr; the line itself goes to the saved descriptor.
    sys.stdout.flush()
    real_stdout = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: limap_b200 has no CPU fallback "
                         "(use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    numa = bind_to_gpu_numa_node(local_rank) if world > 1 else None
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        # NCCL's own log lines (version banner, NCCL_DEBUG output) go to stderr: stdout carries the one JSON line
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    from limap_b200._cabi import NODE_RECORD_DTYPE
    from limap_b200.config import DEFAULT_YAML_TRIANGULATION
    from limap_b200.engine import TriEngine
    from limap_b200 import dist as lmdist

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def reduce_max(x):
        t = torch.tensor([float(x)], device="cuda", dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def reduce_sum(x):
        t = torch.tensor([float(x)], device="cuda", dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t.item())

    def gather_list(x):
        t = torch.tensor([float(x)], device="cuda", dtype=torch.float64)
        if world == 1:
            return [float(x)]
        out = [torch.zeros_like(t) for _ in range(world)]
        dist.all_gather(out, t)
        return [float(o.item()) for o in out]

    scene, per = get_scene(world, rank)
    my_ids = [int(scene.img_ids[v]) for v in range(per * rank, per * (rank + 1))]
    n_rows_rank = scene.n_rows(my_ids)
    cfg = dict(DEFAULT_YAML_TRIANGULATION)
    eng = TriEngine(cfg, device=local_rank)
    eng.ctx.set_stream(torch.cuda.current_stream().cuda_stream)
    eng.upload(scene)
    eng.set_ranges(*scene.ranges)
    flat = {i: scene.flat_matches(i) for i in my_ids}
    for i in my_ids:
        eng.add_image_matches(i, *flat[i])
    eng.set_shard(per * rank, per * (rank + 1))
    eng.set_pipeline_groups(args.value_groups)
    gather = lmdist.NodeGather(eng, world, rank) if world > 1 else None

    def step():
        st = eng.run()
        if gather is not None:
            gather.all_gather()
        return st

    for _ in range(args.warmup):
        st = step()
    if gather is not None:
        gather.check()
    launches0 = eng.stats()["n_kernel_launches"]
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    kernel_ms = []
    e0.record()
    for _ in range(args.steps):
        st = step()
        kernel_ms.append(st["last_node_kernel_ms"])
    e1.record()
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    ms_total = e0.elapsed_time(e1)
    launches = eng.stats()["n_kernel_launches"] - launches0
    n_edges_total = gather.check() if gather is not None else None  # asserts the exchange did not overflow
    if args.dump_outputs and rank == 0:
        dump_outputs(eng, args.dump_outputs, int(scene.line_off[per * rank]), int(scene.line_off[per * (rank + 1)]))
    ms_total = reduce_max(ms_total)
    rows_all = reduce_sum(n_rows_rank)
    value = rows_all * args.steps / (ms_total * 1e-3)
    cand_per_rank = [int(c) for c in gather_list(st["n_candidates"])]

    # ---- roofline of the dominant kernel (fused generate+score), rank 0's launch ----------------
    peak, peak_src = load_peaks()
    km = load_kernel_metrics()
    n_nodes_shard = int(scene.line_off[per * (rank + 1)] - scene.line_off[per * rank])
    alg = algorithmic_bytes(st["n_rows"], n_nodes_shard, scene.n_views, st["n_candidates"], st["n_valid_edges"])
    k_ms = float(np.mean(kernel_ms))
    achieved = alg / (k_ms * 1e-3) / 1e9
    kt = km.get("tri_node_kernel", {})
    same_wl = kt.get("workload") == WORKLOAD and world == 1
    roofline = {"bound": "hbm", "kernel": "tri_node_kernel", "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak, "traffic": kt.get("dram_bytes_per_launch") if same_wl else None,
                "traffic_source": kt.get("source") if same_wl else None, "peak_source": peak_src,
                "algorithmic_bytes_per_launch": alg, "kernel_ms": k_ms,
                "kernel_share_of_step": k_ms * args.steps / ms_total,
                "compute": kt.get("compute"),
                "note": "ALU-bound fp64/fp32 geometry (C^2 pair tests per node); the HBM fraction is low by "
                        "construction (SURVEY.md 8d), `compute` holds the pipe utilisation from the ncu capture"}

    # ---- e2e through the public API with host buffers ------------------------------------------------
    e2e = None
    if not args.no_e2e:
        bsrc, bng, boff, bpairs = scene.bulk_matches(my_ids)
        tp = torch.empty(bpairs.shape, dtype=torch.int32, pin_memory=True)
        tp.numpy()[...] = bpairs
        pinned_pairs = tp.numpy()
        tsegs = torch.empty(scene.segs.shape, dtype=torch.float64, pin_memory=True)  # the 2D segments: pinned as well
        tsegs.numpy()[...] = scene.segs
        scene.segs = tsegs.numpy()
        eng2 = TriEngine(cfg, device=local_rank)
        eng2.ctx.set_stream(torch.cuda.current_stream().cuda_stream)
        eng2.set_pipeline_groups(args.groups)
        eng2.upload(scene)  # (NodeGather reads the node ranges of the shards from the uploaded scene)
        gather2 = lmdist.NodeGather(eng2, world, rank) if world > 1 else None
        h2d = (scene.segs.nbytes + scene.kvec.nbytes + scene.qvec.nbytes + scene.tvec.nbytes +
               scene.line_off.nbytes + pinned_pairs.nbytes)
        nodes_out = torch.empty(int(scene.line_off[-1]) * NODE_RECORD_DTYPE.itemsize, dtype=torch.uint8,
                                pin_memory=True).numpy().view(NODE_RECORD_DTYPE)
        off_out = torch.empty(int(scene.line_off[-1]) + 1, dtype=torch.int64, pin_memory=True).numpy()
        edges_out = torch.empty((max(int(st["n_valid_edges"]) * 2, 1), 2), dtype=torch.int32, pin_memory=True).numpy()

        def e2e_step():
            # public API, bulk form: Init + SetRanges + TriangulateImage(all images) + run + results to host
            eng2.upload(scene)
            eng2.set_ranges(*scene.ranges)
            eng2.add_matches_bulk(bsrc, bng, boff, pinned_pairs)
            eng2.set_shard(per * rank, per * (rank + 1))
            if gather2 is not None:
                s2 = eng2.run()
                gather2.all_gather()
                nodes = eng2.get_nodes(nodes_out)
            else:  # the node records stream into the pinned buffer group by group while the run is going
                s2 = eng2.run(nodes_out=nodes_out)
                nodes = nodes_out
            off, edges = eng2.get_all_valid_edges(off_out, edges_out)
            return s2, nodes.nbytes + off.nbytes + edges.nbytes

        for _ in range(3):
            e2e_step()
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            s2, d2h = e2e_step()
        torch.cuda.synchronize()
        dt = reduce_max(time.perf_counter() - t0)
        e2e = {"value": rows_all * args.steps / dt, "unit": UNIT, "h2d_bytes_per_step": int(h2d),
               "d2h_bytes_per_step": int(d2h), "ms_per_step": 1e3 * dt / args.steps, "pipeline_groups": args.groups,
               "note": "lm_scene_upload + lm_tri_add_matches_bulk (pinned host) + lm_tri_run"
                       + (" + exchange" if world > 1 else "") + (" + lm_tri_get_nodes" if world > 1 else " (node records streamed to the host buffer per pipeline group)") + " + lm_tri_get_all_valid_edges"}
        eng2.close()

    # ---- CPU baseline + parity (rank 0, N=1 only): oracle restatement on a bounded sample -------------------
    cpu = parity = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        from oracle import oracle as orc
        orc.build()
        ncpu = orc.usable_cpus()
        o2 = orc.OracleTri(cfg, threads=ncpu, node_parallel=True)
        o2.upload(scene)
        o2.set_ranges(*scene.ranges)
        t0 = time.perf_counter()
        done = []
        for i in my_ids:
            o2.add_image_matches(i, *flat[i])
            done.append(i)
            if time.perf_counter() - t0 > 0.7 * args.cpu_seconds:
                break
        dt2 = time.perf_counter() - t0
        cpu = {"value": o2.rows_tested() / dt2, "unit": UNIT, "cores": ncpu, "kind": "port", "host_cpus": ncpu,
               "schedule": "OpenMP over the 2D lines of an image (identical results to the reference's schedule)",
               "sample": f"first {len(done)} source images of the scene ({o2.rows_tested()} rows, {dt2:.1f} s)"}
        try:
            parity = tri_parity(eng, o2, done)
            parity["checked_rows"] = int(o2.rows_tested())
            if len(done) == len(my_ids):  # the whole scene went through the oracle: ComputeLineTracks on both sides
                t0 = time.perf_counter()
                gt = eng.build_tracks()
                t_cold = time.perf_counter() - t0  # first call: device scratch is allocated
                t0 = time.perf_counter()
                gt = eng.build_tracks()
                t_gpu = time.perf_counter() - t0
                t0 = time.perf_counter()
                ot = o2.build_tracks()
                t_cpu = time.perf_counter() - t0
                mem = lambda tr: sorted(tuple(sorted(zip(tr["img_ids"][a:b].tolist(), tr["line_ids"][a:b].tolist())))
                                        for a, b in zip(tr["track_off"][:-1], tr["track_off"][1:]))
                parity["tracks"] = {"n_tracks": len(gt["track_off"]) - 1, "membership_identical": mem(gt) == mem(ot),
                                    "compute_line_tracks_ms": 1e3 * t_gpu, "compute_line_tracks_first_call_ms": 1e3 * t_cold, "cpu_port_ms": 1e3 * t_cpu,
                                    "note": "run_clustering + greedy labels + aggregation: edge weights on the device, "
                                            "union-find on the host (sequential by definition)"}
        except Exception as e:  # the check must never cost the bench line
            parity = {"error": str(e)}
        del o2
        try:
            make, kind = reference_impl()
            cores = pick_cpu_threads(scene, make)
            o = make(cfg, cores)
            o.upload(scene)
            o.set_ranges(*scene.ranges)
            t0 = time.perf_counter()
            n_img = 0
            for i in my_ids:
                o.add_image_matches(i, *flat[i])
                n_img += 1
                if time.perf_counter() - t0 > 0.3 * args.cpu_seconds:
                    break
            dt = time.perf_counter() - t0
            cpu["reference_schedule"] = {
                "value": o.rows_tested() / dt, "cores": cores, "kind": kind,
                "sample": f"first {n_img} source images ({o.rows_tested()} rows, {dt:.1f} s), "
                          + ("the reference's own sources compiled unchanged (oracle/_ref)" if kind == "reference"
                             else "the restatement with the reference's loop structure")
                          + ", OpenMP over connections / candidates of one node, fastest thread count of 1/8/32/all"}
            del o
        except Exception as e:
            cpu["reference_schedule"] = {"error": str(e)}

    extra = {}
    if not args.no_lm:
        extra = side_legs(args, eng, rank, world, local_rank, barrier, reduce_max, reduce_sum, km, peak)

    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": ms_total / args.steps, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                "config": {"workload": WORKLOAD, "V": 100 * world, "L": 1000, "N": 20, "K": 10,
                           "blocks": world, "rows_per_step": int(rows_all),
                           "candidates_per_step_per_rank": cand_per_rank,
                           "valid_connections_rank0": int(st["n_valid_edges"]),
                           "exchanged_directed_edges": n_edges_total,
                           "pairs": {"past_3d_gates": int(st["n_pairs_gated"]), "scored_exact_fp64": int(st["n_pairs_exact"])},
                           "parallelism": f"source-image shards x{world}"
                                          + (", one all-gather of node records + valid connections per step" if world > 1 else ""),
                           "host_cpus_bound_rank0": numa, "pipeline_groups_resident_leg": args.value_groups,
                           "l2": "inputs larger than L2 (match rows + sort buffers > 126 MB per step)"},
                "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches), "roofline": roofline,
                "cpu_baseline": cpu, "parity": parity}
        line.update(extra)
        real_stdout.write(json.dumps(line) + "\n")
        real_stdout.flush()
    if world > 1:
        dist.destroy_process_group()


def side_legs(args, eng, rank, world, local_rank, barrier, reduce_max, reduce_sum, km, peak):
    """M2 (line BA), remerge, J-Linkage and the configs[2] sweep; every rank takes part, rank 0 reports."""
    import torch
    from limap_b200 import dist as lmdist
    out = {}
    cpu_ok = rank == 0 and world == 1 and not args.no_cpu_baseline

    # ---- M2: line-BA LM iterations/s (configs[3]: 10k tracks x 30 supporting views per GPU) --------------------
    # N > 1: ONE problem of 10k*N tracks, dealt to the ranks by support count, refined lines all-gathered
    # (dist.solve_line_ba_sharded; block-separable with constant cameras).
    from limap_b200.engine import BAEngine
    from limap_b200.synth import make_tracks
    T = 10000 * world
    ts = make_tracks(T=T, S=30, V=300, seed=1237)
    ba = BAEngine(ctx=eng.ctx)
    views, first_idx = np.unique(ts.img_ids, return_index=True)
    remap = np.zeros(int(views.max()) + 1, np.int32)
    remap[views] = np.arange(len(views), dtype=np.int32)
    def pin(x):  # e2e inputs live in pinned host memory (the copies inside lm_ba_solve are then real async DMA)
        x = np.ascontiguousarray(x)
        t = torch.empty(x.shape, dtype=torch.from_numpy(x[:0].copy()).dtype, pin_memory=True)
        t.numpy()[...] = x
        return t.numpy()
    a = tuple(pin(x) for x in (ts.kvec[first_idx], ts.qvec[first_idx], ts.tvec[first_idx], ts.sup_off.astype(np.int64),
                               remap[ts.img_ids].astype(np.int32), ts.segs, ts.line3d, ts.line_init))
    k_ms = []

    def solve_once():
        if world == 1:
            o = ba.solve(*a, max_num_iterations=100)
            k_ms.append(o["stats"]["solve_ms"])
            return int(o["stats"]["total_iterations"])

        def solve(*aa, **kw):
            o = ba.solve(*aa, **kw)
            k_ms.append(o["stats"]["solve_ms"])
            return o
        o = lmdist.solve_line_ba_sharded(solve, *a, rank=rank, world=world, max_num_iterations=100)
        return int(o["iters"][:, 0].sum())

    for _ in range(2):
        solve_once()
    k_ms.clear()
    barrier()
    t0 = time.perf_counter()
    iters = 0
    for _ in range(args.steps):
        iters += solve_once()
    torch.cuda.synchronize()
    dt = reduce_max(time.perf_counter() - t0)
    kern_s = reduce_max(float(np.sum(k_ms)) * 1e-3)
    its = iters // args.steps
    klm = km.get("lm_refine_kernel", {})
    b_lm = T * (30 * 20 + 24 + 24)  # SURVEY.md 8(d): B_lm = T (S 20 + 24 in + 24 out), once per solve
    f_lm = its * 30 * 400.0          # F_lm = iterations x S x F_blk (400 flop per block evaluation)
    kms = kern_s / args.steps
    lm_ba = {"metric": "line-BA LM iters/sec", "unit": "track LM iterations/s",
             "config": {"workload": "ba10k", "tracks": T, "tracks_per_gpu": 10000, "supports": 30,
                        "max_num_iterations": 100,
                        "parallelism": "one problem, tracks dealt by support count, lines all-gathered" if world > 1 else "1 GPU"},
             "value_kernel": float(iters / kern_s),
             "e2e": {"value": float(iters / dt),
                     "note": "lm_ba_solve from host arrays: H2D, solve, segment cut, D2H" + (", all-gather" if world > 1 else "")},
             "kernel_ms": float(1e3 * kms), "iterations_per_solve": int(its), "dtype": "f64",
             "roofline": {"bound": "hbm", "kernel": "lm_refine_kernel", "achieved": b_lm / world / kms / 1e9, "peak": peak,
                          "unit": "GB/s", "frac": b_lm / world / kms / 1e9 / peak,
                          "traffic": klm.get("dram_bytes_per_launch") if world == 1 else None,
                          "algorithmic_bytes_per_launch": b_lm // world,
                          "flops": {"achieved_tflops": f_lm / world / kms / 1e12, "nominal_fp64_tflops": FP64_NOMINAL_TFLOPS,
                                    "frac": f_lm / world / kms / 1e12 / FP64_NOMINAL_TFLOPS,
                                    "per_block_evaluation": 400},
                          "compute": klm.get("compute"),
                          "note": "latency/ALU-bound fp64 iteration chain; the working set is read once per solve"}}
    if cpu_ok:
        from oracle import oracle as orc
        sub = make_tracks(T=1500, S=30, V=300, seed=1237)
        best = None
        for th in sorted({min(8, orc.usable_cpus()), orc.usable_cpus()}):
            t0 = time.perf_counter()
            o = orc.refine_tracks(sub, max_num_iterations=100, threads=th)
            v = float(o["iters"][:, 0].sum() / (time.perf_counter() - t0))
            if best is None or v > best[0]:
                best = (v, th)
        lm_ba["cpu_baseline"] = {"value": best[0], "unit": "track LM iterations/s", "cores": best[1], "kind": "port",
                                 "sample": "1500 tracks x 30 supports, Ceres-style LM restatement, OpenMP over tracks"}
    out["lm_ba"] = lm_ba

    # ---- remerge pair test (SURVEY.md 8(f) rank 1): all-pairs check_connection over 1e5 track lines, rank 0 ----
    if rank == 0:
        from limap_b200.config import LINKER3D_DEFAULTS, make_linker
        from limap_b200.engine import MergeEngine
        from limap_b200.synth import make_track_lines
        lk = dict(score_th=0.5, th_angle=5.0, th_overlap=0.001, th_smartoverlap=0.1, th_smartangle=1.0, th_perp=1.0,
                  th_innerseg=1.0)  # cfgs/triangulation/default.yaml:99-108
        Tm = 100000
        TL = make_track_lines(Tm, dup_frac=0.3, seed=1, extent=60.0)
        me = MergeEngine(ctx=eng.ctx)
        act = np.ones(Tm, np.uint8)
        k_ms, w_ms = [], []
        for it in range(2 + args.steps):
            t0 = time.perf_counter()
            _, ng, ne = me.remerge_labels(TL, act, make_linker(LINKER3D_DEFAULTS, lk))
            if it >= 2:
                w_ms.append((time.perf_counter() - t0) * 1e3)
                k_ms.append(me.stats()["last_remerge_kernel_ms"])
        pairs = Tm * (Tm - 1) / 2
        krm = km.get("remerge_pairs_kernel", {})
        kms = float(np.mean(k_ms)) * 1e-3
        b_rm = Tm * (56 + 32) + 8 * ne  # track lines + gate records read once, edge list written
        remerge = {"metric": "remerge pair tests/sec", "unit": "track pairs/s",
                   "config": {"workload": "remerge100k", "tracks": Tm, "groups": ng, "edges": ne,
                              "pairs_past_fp32_gate": int(me.stats()["n_pairs_gated"])},
                   "value_kernel": pairs / kms, "kernel_ms": 1e3 * kms,
                   "e2e": {"value": pairs / (float(np.mean(w_ms)) * 1e-3),
                           "note": "lm_remerge_labels from host arrays: H2D, pair kernel, edge list D2H, host union-find"},
                   "dtype": "f32 gate + f64 check",
                   "roofline": {"bound": "hbm", "kernel": "remerge_pairs_kernel", "achieved": b_rm / kms / 1e9, "peak": peak,
                                "unit": "GB/s", "frac": b_rm / kms / 1e9 / peak, "traffic": krm.get("dram_bytes_per_launch"),
                                "algorithmic_bytes_per_launch": int(b_rm), "compute": krm.get("compute"),
                                "note": "O(T^2) fp32 pair gates on O(T) bytes: bound by the fp32 issue rate, not HBM"}}
        if cpu_ok:
            from oracle import oracle as orc
            Ts = 20000
            sub = make_track_lines(Ts, dup_frac=0.3, seed=1, extent=60.0)
            t0 = time.perf_counter()
            orc.remerge_labels(sub, np.ones(Ts, np.uint8), lk, threads=orc.usable_cpus())
            dtc = time.perf_counter() - t0
            remerge["cpu_baseline"] = {"value": Ts * (Ts - 1) / 2 / dtc, "unit": "track pairs/s",
                                       "cores": orc.usable_cpus(), "kind": "port",
                                       "sample": f"{Ts} tracks, all pairs, OpenMP over tracks ({dtc:.2f} s)"}
        out["remerge"] = remerge

    # ---- J-Linkage VP detection (a18; configs[4] slice: 1000 images x 300 segments x 5000 hypotheses per GPU) ------
    from limap_b200.synth import make_vp_images
    from limap_b200.vplib import JLinkageDetector
    n_img = 1000 * world
    imgs = make_vp_images(n_img, 300, seed=77)
    det = JLinkageDetector(dict(min_num_supports=10, min_length=40, inlier_threshold=1.0), device=local_rank, seed=7)
    mine = lmdist.partition_by_cost([len(s) for s in imgs], world)[rank]
    my_imgs = [imgs[i] for i in mine]
    det.detect_batch(my_imgs[:64], image_index=mine[:64])  # warm-up
    barrier()
    kj_ms = []
    t0 = time.perf_counter()
    for _ in range(args.steps):  # one step = every image once
        if world == 1:
            res = det.detect_batch(my_imgs, image_index=mine)
            n_vps = sum(r.count_vps() for r in res)
        else:
            res = lmdist.detect_vps_sharded(det.detect_batch, imgs, rank, world)
            n_vps = sum(len(v) for v in res[1])
        kj_ms.append(det.stats()["kernel_ms"])  # kernel time of this rank's last detect_batch call
    torch.cuda.synchronize()
    dt = reduce_max(time.perf_counter() - t0) / args.steps
    kj = reduce_max(float(np.mean(kj_ms))) * 1e-3
    kjl = km.get("jlinkage_kernel", {})
    b_j = 1000 * 300 * (16 + 4)  # per GPU: float4 segment in, label out
    jl = {"metric": "J-Linkage images/sec", "unit": "images/s", "steps": args.steps,
          "config": {"workload": "rome16k-slice", "images": n_img, "segments_per_image": 300, "hypotheses": 5000,
                     "vps_found": int(n_vps),
                     "parallelism": "images dealt by segment count, labels + VPs all-gathered" if world > 1 else "1 GPU"},
          "value_kernel": n_img / kj, "kernel_ms": 1e3 * kj,
          "e2e": {"value": n_img / dt, "note": "lm_vp_detect from host arrays: filter, H2D, clustering kernel, D2H, host VP fit"},
          "dtype": "f32 consensus + integer set algebra",
          "roofline": {"bound": "hbm", "kernel": "jlinkage_kernel", "achieved": b_j / kj / 1e9, "peak": peak, "unit": "GB/s",
                       "frac": b_j / kj / 1e9 / peak, "traffic": kjl.get("dram_bytes_per_launch") if world == 1 else None,
                       "algorithmic_bytes_per_launch": b_j, "compute": kjl.get("compute"),
                       "note": "preference matrix (300 x 5000 bits) and the merge loop live in shared memory / L2: "
                               "bound by ALU + shared-memory bit operations"}}
    if cpu_ok:
        from oracle import oracle as orc
        ns = 2 * orc.usable_cpus()
        off = np.concatenate([[0], np.cumsum([len(s) for s in imgs[:ns]])]).astype(np.int64)
        t0 = time.perf_counter()
        lab, _, _ = orc.detect_vps(off, np.concatenate(imgs[:ns], 0), min_length=40, inlier_threshold=1.0,
                                   min_num_supports=10, seed=7, threads=orc.usable_cpus())
        dtc = time.perf_counter() - t0
        same = all(np.array_equal(np.asarray(res[i].labels, np.int32), lab[off[i]:off[i + 1]]) for i in range(ns))
        jl["cpu_baseline"] = {"value": ns / dtc, "unit": "images/s", "cores": orc.usable_cpus(), "kind": "port",
                              "sample": f"first {ns} images, OpenMP over images ({dtc:.2f} s)",
                              "labels_identical_to_gpu": bool(same)}
    out["jlinkage"] = jl

    # ---- configs[2]: synthetic 500 views x 400 lines x 40 neighbours, STRONG scaling of one fixed scene -----------
    from limap_b200.config import DEFAULT_YAML_TRIANGULATION
    from limap_b200.engine import TriEngine
    from limap_b200.synth import CONFIGS, make_scene
    c2 = dict(CONFIGS["sweep500"])
    w_rows = None
    sc0 = make_scene(match_views=[], **c2)  # cameras + segments + neighbours (cheap); matches only for the shard
    V2, L2, N2, K2 = c2["V"], c2["L"], c2["N"], c2["K"]
    w_rows = np.array([len(sc0.neighbors[int(i)]) * (sc0.line_off[v + 1] - sc0.line_off[v]) * K2
                       for v, i in enumerate(sc0.img_ids)], np.float64)
    shards = lmdist.partition_views(w_rows, world)
    vb, ve = shards[rank]
    sc2 = make_scene(match_views=range(vb, ve), **c2)
    e3 = TriEngine(dict(DEFAULT_YAML_TRIANGULATION), device=local_rank)
    e3.ctx.set_stream(torch.cuda.current_stream().cuda_stream)
    e3.upload(sc2)
    e3.set_ranges(*sc2.ranges)
    ids3 = [int(sc2.img_ids[v]) for v in range(vb, ve)]
    e3.add_matches_bulk(*sc2.bulk_matches(ids3))
    e3.set_shard(vb, ve)
    g3 = lmdist.NodeGather(e3, world, rank, shards=shards) if world > 1 else None
    nst = args.steps
    for _ in range(2):
        s3 = e3.run()
        if g3 is not None:
            g3.all_gather()
    if g3 is not None:
        g3.check()
    barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(nst):
        s3 = e3.run()
        if g3 is not None:
            g3.all_gather()
    ev1.record()
    barrier()
    ms3 = reduce_max(ev0.elapsed_time(ev1)) / nst
    if g3 is not None:
        g3.check()
    rows3 = reduce_sum(s3["n_rows"])
    out["sweep500"] = {"metric": METRIC, "unit": UNIT, "scaling": "strong",
                       "config": {"workload": "sweep500", "V": V2, "L": L2, "N": N2, "K": K2, "rows": int(rows3),
                                  "shards": [list(map(int, s)) for s in shards],
                                  "candidates_total": int(reduce_sum(s3["n_candidates"]))},
                       "value": rows3 / (ms3 * 1e-3), "ms_per_step": ms3, "steps": nst,
                       "node_kernel_ms_rank0": float(s3["last_node_kernel_ms"])}
    e3.close()
    return out


if __name__ == "__main__":
    main()
