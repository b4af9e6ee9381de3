"""Pins the oracle (oracle/*.h, the restatement every GPU parity test compares against) and the Python mirror to the
REFERENCE'S OWN COMPILED CODE: the reference's hot-path sources built unchanged into oracle/_ref/liblimap_ref.so
(oracle/Makefile target `ref`; Eigen / COLMAP / glog / PoseLib come from the header shims in oracle/ref_shim/).

What the compiled reference returned is stored in tests/golden/ref/<test>.npz (tests/golden/make_ref_golden.py runs this
module with LIMAP_REF_RECORD=1 against the library); every test regenerates its seeded inputs, runs the oracle / mirror
on them and compares with the stored reference outputs, so the suite needs neither the reference tree nor the library.
Floating-point outputs are stored for a fixed sample of each test's inputs (the first inputs of its seeded stream, or
seeded node / track samples), integer outputs in full.

  * whole pipeline: limap::triangulation::GlobalLineTriangulator (Init -> TriangulateImage -> ComputeLineTracks) against
    OracleTri on seeded scenes and every configuration family the GPU tests use -- candidate counts, best candidates,
    valid connections, graph-ordered track membership bit-exact; candidate lists, scores and coordinates to 1e-9;
  * function level: compute_epipolar_IoU, triangulate_line (plane pair and endpoints), triangulate_line_with_direction,
    LineLinker2d/3d::compute_score, Line3d::sensitivity / computeUncertainty, CameraView::projection / ray_direction,
    Aggregator::aggregate_line3d_list, MinimalInfiniteLine3d, GetLineSegmentFromInfiniteLine3d, CheckReprojection /
    CheckSensitivity / overlap, RemergeLineTracks;
  * fixture consistency: the frozen golden fixtures (tests/golden/hotpath) agree with what the reference's compiled code
    computed on their inputs."""
import ctypes as C
import os

import numpy as np
import pytest

from limap_b200.config import DEFAULT_YAML_TRIANGULATION
from limap_b200.synth import make_scene

from oracle import oracle as orc
from oracle import ref
from ref_golden import reference as _reference

TOL = 1e-9


def _tri(cls, sc, cfg, exhaustive=False, ranges=True, vp=None):
    t = cls(cfg, threads=1)
    t.upload(sc)
    if ranges:
        t.set_ranges(*sc.ranges)
    if vp is not None:
        t.set_vps(vp, sc.img_ids, sc.line_off)
    for i in sc.img_ids:
        if exhaustive:
            t.add_image_exhaustive(int(i), sc.neighbors[int(i)])
        else:
            t.add_image_matches(int(i), *sc.flat_matches(int(i)))
    return t


N_NODES, N_CAND_NODES, N_TRACKS = 16, 3, 16  # stored samples of the floating-point outputs of one scene


def _tri_outputs(t, img_ids, sample_seed):
    """What a triangulator answers on a scene. In full: every node's candidate count and best candidate ids, every valid
    connection (sorted per node: the reference keeps them in score order, run_clustering reads them as a set) and the
    track membership in graph order. Sampled: best candidates of N_NODES seeded nodes, whole candidate lists of the
    first N_CAND_NODES of them, lines of the first N_TRACKS tracks."""
    best, ng, nc, eoff, edges, where = [], [], [], [0], [], []
    for i in img_ids:
        l, g, c = t.get_best(int(i))
        best.append(l); ng.append(g); nc.append(c)
        where += [(int(i), k) for k in range(len(c))]
        off, e = t.get_valid_edges(int(i))
        for k in range(len(off) - 1):
            ee = sorted(map(tuple, e[off[k]:off[k + 1]]))
            edges.extend(ee)
            eoff.append(eoff[-1] + len(ee))
    best, ng, nc = np.concatenate(best), np.concatenate(ng), np.concatenate(nc)
    nodes = np.sort(np.random.default_rng(sample_seed).choice(len(nc), min(len(nc), N_NODES), replace=False))
    cand_off, cand_ng, cand_line = [0], [], []
    for n in nodes[:N_CAND_NODES]:
        cl, cg = t.get_cands_node(*where[n])
        cand_ng.append(cg); cand_line.append(cl)
        cand_off.append(cand_off[-1] + len(cg))
    tr = t.build_tracks()
    return dict(n_cand=nc, best_ng=ng, edge_off=np.asarray(eoff, np.int64), edges=np.asarray(edges, np.int32).reshape(-1, 2),
                nodes=nodes, best_line=best[nodes], cand_off=np.asarray(cand_off, np.int64),
                cand_ng=np.concatenate(cand_ng).reshape(-1, 2), cand_line=np.concatenate(cand_line).reshape(-1, 10),
                track_off=tr["track_off"], track_img=tr["img_ids"], track_line_id=tr["line_ids"],
                track_line=tr["track_line"][:N_TRACKS])


def _compare_tri(r, o, line3d, end_tol, score_tol):
    """r: the reference's _tri_outputs, o: the oracle's; line3d: the oracle's per-support 3D lines (ties below)."""
    assert np.array_equal(o["n_cand"], r["n_cand"]), "candidate counts differ"
    has = r["n_cand"] > 0
    assert np.array_equal(o["best_ng"][has], r["best_ng"][has]), "best candidate ids differ"
    assert np.array_equal(o["nodes"], r["nodes"])
    h = r["n_cand"][r["nodes"]] > 0
    for a, b in ((o["best_line"][h], r["best_line"][h]), (o["cand_line"], r["cand_line"])):
        assert np.abs(a[:, :9] - b[:, :9]).max(initial=0) <= end_tol
        assert np.abs(a[:, 9] - b[:, 9]).max(initial=0) <= score_tol
    for k in ("edge_off", "edges", "cand_off", "cand_ng", "track_off", "track_img", "track_line_id"):
        assert np.array_equal(o[k], r[k]), k  # valid connections, candidate lists, tracks in graph order: bit-exact
    for k, (a, b) in enumerate(zip(o["track_line"], r["track_line"])):
        d = min(np.abs(a[:6] - b[:6]).max(), np.abs(a[:6] - np.concatenate([b[3:6], b[:3]])).max())
        ta, tb = r["track_off"][k], r["track_off"][k + 1]
        if d > end_tol and tb - ta < 4:
            # aggregate_line3d_list_takebest keeps the first strict maximum of the node scores; two nodes of a track that
            # triangulate each other carry the same infinite line and their scores tie to the last bits (parity_utils)
            sc = line3d[ta:tb, 9]
            tied = [m for m in range(tb - ta) if sc[m] >= sc.max() * (1 - 1e-9)]
            if len(tied) > 1:
                d = min(d, min(np.abs(b[:6] - line3d[ta + m, :6]).max() for m in tied))
        assert d <= end_tol, (k, d)
        assert abs(a[6] - b[6]) <= end_tol
    return dict(candidates=int(r["n_cand"].sum()), valid_edges=len(r["edges"]), tracks=len(r["track_off"]) - 1)


def _cfg(**kw):
    c = dict(DEFAULT_YAML_TRIANGULATION, debug_mode=True)
    c.update(kw)
    return c


def _vps(sc, seed):
    rng = np.random.default_rng(seed)
    out = {}

    class R:
        pass
    for v, i in enumerate(sc.img_ids):
        L = int(sc.line_off[v + 1] - sc.line_off[v])
        q = rng.normal(size=(3, 3))
        q[:, :2] *= 1000.0
        q /= np.linalg.norm(q, axis=1, keepdims=True)
        lab = rng.integers(0, 3, L)
        lab[rng.random(L) < 0.4] = -1
        r = R()
        r.labels, r.vps = lab.astype(np.int32), q
        out[int(i)] = r
    return out


CASES = {
    "default_yaml": (dict(V=8, L=120, N=5, K=6, seed=201), {}, {}),
    "cpp_defaults_outer_edge_filter": (dict(V=8, L=120, N=5, K=5, seed=202), None, {}),
    "asset_units_gaps_shuffled": (dict(V=8, L=100, N=5, K=4, seed=203, scale=100.0, id_stride=7, shuffle_rows=True), {}, {}),
    "mixed_cameras": (dict(V=8, L=100, N=5, K=5, seed=204, camera_mix=True), {}, {}),
    "endpoints_halfpix_no_ranges": (dict(V=6, L=80, N=4, K=4, seed=205), dict(use_endpoints_triangulation=True, add_halfpix=True), dict(ranges=False)),
    "max_valid_conns": (dict(V=6, L=60, N=5, K=8, seed=206), dict(max_valid_conns=3), {}),
    "exhaustive": (dict(V=5, L=40, N=3, K=2, seed=207), {}, dict(exhaustive=True)),
    "vp_proposals": (dict(V=6, L=60, N=4, K=3, seed=208), dict(use_vp=True), dict(vp=9)),
    "innerseg_2d_linker": (dict(V=6, L=80, N=4, K=4, seed=209), dict(linker2d_config=dict(use_innerseg=True, th_innerseg=3.0)), {}),
}


@pytest.mark.parametrize("name", sorted(CASES))
def test_whole_pipeline_oracle_equals_compiled_reference(name):
    kw, over, run = CASES[name]
    sc = make_scene(**kw)
    cfg = dict(debug_mode=True) if over is None else _cfg(**over)
    run = dict(run)
    if "vp" in run:
        run["vp"] = _vps(sc, run["vp"])
    seed = kw["seed"]
    o = _tri(orc.OracleTri, sc, cfg, **run)
    r = _reference(f"pipeline_{name}", lambda: _tri_outputs(_tri(ref.RefTri, sc, cfg, **run), sc.img_ids, seed))
    st = _compare_tri(r, _tri_outputs(o, sc.img_ids, seed), o.build_tracks()["line3d"],
                      1e-7 * (100.0 if kw.get("scale") else 1.0), 1e-9)
    assert st["candidates"] > 200 and st["valid_edges"] > 20 and st["tracks"] > 5


# ---- function level --------------------------------------------------------------------------------------------
def _rand_cam(rng, mixed=True):
    f = rng.uniform(400, 900)
    model = int(rng.integers(0, 2)) if mixed else 0
    fy = f * rng.uniform(0.9, 1.1) if model == 1 else f
    q = rng.normal(size=4)
    q /= np.linalg.norm(q)
    return orc.cam_array(model, [f, fy, rng.uniform(300, 500), rng.uniform(200, 400)], q, rng.normal(size=3) * 3)


def _look_at_cam(rng, target, dist):
    from limap_b200.synth import _rot_to_quat
    c = target + dist * (lambda v: v / np.linalg.norm(v))(rng.normal(size=3))
    z = (target - c) / np.linalg.norm(target - c)
    x = np.cross(z, rng.normal(size=3))
    x /= np.linalg.norm(x)
    R = np.stack([x, np.cross(z, x), z], 0)
    f = rng.uniform(500, 800)
    return orc.cam_array(0, [f, f, 400, 300], _rot_to_quat(R), -R @ c), R, -R @ c, f


def _proj(R, t, f, X):
    Xc = R @ X + t
    return Xc[:2] / Xc[2] * f + np.array([400.0, 300.0])


def _pairs_of_views(rng, n):
    """(l1, cam1, l2, cam2): projections of a random 3D segment into two looking-at cameras, with pixel noise."""
    out = []
    for _ in range(n):
        X0, X1 = rng.uniform(-2, 2, 3), rng.uniform(-2, 2, 3)
        c1, R1, t1, f1 = _look_at_cam(rng, (X0 + X1) / 2, rng.uniform(6, 12))
        c2, R2, t2, f2 = _look_at_cam(rng, (X0 + X1) / 2, rng.uniform(6, 12))
        l1 = np.concatenate([_proj(R1, t1, f1, X0), _proj(R1, t1, f1, X1)]) + rng.normal(scale=1.0, size=4)
        l2 = np.concatenate([_proj(R2, t2, f2, X0), _proj(R2, t2, f2, X1)]) + rng.normal(scale=1.0, size=4)
        out.append((np.ascontiguousarray(l1), c1, np.ascontiguousarray(l2), c2))
    return out


def _close(a, b, tol=TOL):
    a, b = np.asarray(a, float), np.asarray(b, float)
    return np.all((np.abs(a - b) <= tol * (1 + np.abs(b))) | (np.isnan(a) & np.isnan(b)))


def _two_view(L, pre, pairs, dirs):
    """compute_epipolar_IoU, triangulate_line (by planes, by endpoints), triangulate_line_with_direction on each pair."""
    f = lambda n: getattr(L, pre + n)
    f("compute_epipolar_IoU").restype = C.c_double
    f("compute_epipolar_IoU").argtypes = [C.c_void_p] * 4
    f("triangulate_line_with_direction").argtypes = [C.c_void_p] * 6
    p = orc._p
    out = np.zeros((len(pairs), 28))
    for k, ((l1, c1, l2, c2), d) in enumerate(zip(pairs, dirs)):
        out[k, 0] = f("compute_epipolar_IoU")(p(l1), p(c1), p(l2), p(c2))
        for by_end in (0, 1):
            f("triangulate_line")(p(l1), p(c1), p(l2), p(c2), by_end, p(out[k, 1 + 9 * by_end:10 + 9 * by_end]))
        f("triangulate_line_with_direction")(p(l1), p(c1), p(l2), p(c2), p(d), p(out[k, 19:28]))
    return out


def test_two_view_functions_on_random_pairs():
    rng = np.random.default_rng(301)
    pairs = _pairs_of_views(rng, 30)
    dirs = []
    for _ in pairs:
        d = rng.normal(size=3)
        dirs.append(d / np.linalg.norm(d))
    a = _two_view(orc.lib(), "orc_", pairs, dirs)
    b = _reference("two_view", lambda: dict(out=_two_view(ref.lib(), "ref_", pairs, dirs)))["out"]
    assert _close(a[:, 0], b[:, 0])
    n_ok = 0
    for c, tol in ((1, 1e-8), (10, 1e-8), (19, 1e-8)):
        assert np.array_equal(a[:, c + 8], b[:, c + 8])  # score: 1 on success, -1 on failure -- the same decision
        ok = b[:, c + 8] > 0
        assert _close(a[ok, c:c + 9], b[ok, c:c + 9], tol)
        n_ok += int(ok.sum()) if c < 19 else 0
    assert n_ok > len(pairs)


def _camera_line3d(L, pre, inputs):
    for f in ("line3d_sensitivity", "line3d_uncertainty"):
        getattr(L, pre + f).restype = C.c_double
    getattr(L, pre + "line3d_sensitivity").argtypes = [C.c_void_p] * 2
    getattr(L, pre + "line3d_uncertainty").argtypes = [C.c_void_p, C.c_void_p, C.c_double]
    getattr(L, pre + "ray_direction").argtypes = [C.c_void_p] * 3
    p = orc._p
    out = np.zeros((len(inputs), 7))
    for k, (cam, X, px, l3) in enumerate(inputs):
        getattr(L, pre + "project_point")(p(cam), p(X), p(out[k, 0:2]))
        getattr(L, pre + "ray_direction")(p(cam), p(px), p(out[k, 2:5]))
        out[k, 5] = getattr(L, pre + "line3d_sensitivity")(p(l3), p(cam))
        out[k, 6] = getattr(L, pre + "line3d_uncertainty")(p(l3), p(cam), 2.0)
    return out


def test_camera_and_line3d_functions():
    rng = np.random.default_rng(302)
    inputs = []
    for _ in range(100):
        cam = _rand_cam(rng)
        X = rng.normal(size=3) * 5
        px = rng.uniform(0, 800, 2)
        l3 = np.concatenate([rng.normal(size=6) * 3, rng.uniform(1, 9, 2), [0.1]])
        inputs.append((cam, X, px, l3))
    a = _camera_line3d(orc.lib(), "orc_", inputs)
    b = _reference("camera_line3d", lambda: dict(out=_camera_line3d(ref.lib(), "ref_", inputs)))["out"]
    assert _close(a[:, 0:2], b[:, 0:2], 1e-9)
    assert _close(a[:, 2:5], b[:, 2:5], 1e-12)
    assert _close(a[:, 5], b[:, 5], 1e-9)
    assert _close(a[:, 6], b[:, 6], 1e-12)


def test_linker_scores_on_random_pairs():
    rng = np.random.default_rng(303)
    variants = [dict(), dict(use_perp=1, use_innerseg=0), dict(use_scaleinv=1, use_overlap=0, use_innerseg=0),
                dict(use_innerseg=1, use_perp=1, use_scaleinv=1), dict(use_angle=0, use_smartangle=0)]
    inputs = []
    for k in range(500):
        v = dict(variants[k % len(variants)])
        v.update(score_th=0.5, th_angle=rng.uniform(3, 12), th_overlap=rng.uniform(0.01, 0.2), th_smartoverlap=0.25,
                 th_smartangle=1.0, th_perp=rng.uniform(0.5, 3), th_innerseg=rng.uniform(0.5, 3), th_scaleinv=0.05)
        # 2D: a segment and a noisy, shifted, maybe flipped copy
        a = rng.uniform(0, 600, 4)
        d = (a[2:] - a[:2]) / np.linalg.norm(a[2:] - a[:2])
        s = rng.uniform(-0.5, 0.5, 2) * np.linalg.norm(a[2:] - a[:2])
        b = np.concatenate([a[:2] + d * s[0], a[2:] + d * s[1]]) + rng.normal(scale=rng.choice([0.3, 3.0]), size=4)
        if rng.random() < 0.5:
            b = b[[2, 3, 0, 1]]
        # 3D: start3, end3, depths2, uncertainty
        A = np.concatenate([rng.normal(size=6) * 2, rng.uniform(2, 9, 2), [rng.uniform(0.01, 0.2)]])
        dd = (A[3:6] - A[:3]) / np.linalg.norm(A[3:6] - A[:3])
        B = A.copy()
        B[:3] += dd * rng.uniform(-0.5, 0.5) + rng.normal(scale=rng.choice([0.005, 0.1]), size=3)
        B[3:6] += dd * rng.uniform(-0.5, 0.5) + rng.normal(scale=rng.choice([0.005, 0.1]), size=3)
        inputs.append((ref.linker_cfg(v), np.ascontiguousarray(a), np.ascontiguousarray(b), A, B))

    def scores(L, pre):
        p = orc._p
        return np.array([[getattr(L, pre + "score_2d")(C.byref(cfg), p(a), p(b)),
                          getattr(L, pre + "score_3d")(C.byref(cfg), p(A), p(B))] for cfg, a, b, A, B in inputs])
    x = scores(orc.lib(), "orc_")
    y = _reference("linker_scores", lambda: dict(out=scores(ref.lib(), "ref_")))["out"]
    assert _close(x, y, 1e-9)
    assert (y[:, 1] > 0).sum() > len(inputs) // 10


def test_aggregator_minimal_line_and_segment_cut():
    rng = np.random.default_rng(304)
    # aggregate_line3d_list: groups of 1..12 noisy copies of a segment
    sizes = rng.integers(1, 13, 20000)
    off = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
    base = rng.normal(size=(len(sizes), 6)) * 3
    lines = np.repeat(base, sizes, 0) + rng.normal(scale=0.02, size=(off[-1], 6))
    lines = np.concatenate([lines, rng.uniform(0.01, 0.3, (off[-1], 1))], 1)
    scores = rng.uniform(0, 5, off[-1])
    groups = {}
    for no in (0, 2):
        ok = sizes * 2 - 1 - no >= no
        o2 = np.concatenate([[0], np.cumsum(sizes[ok])]).astype(np.int64)
        sel = np.repeat(ok, sizes)
        keep = np.sort(np.random.default_rng(no).choice(len(o2) - 1, 32, replace=False))
        groups[no] = (o2, lines[sel], scores[sel], keep)
    # MinimalInfiniteLine3d round trip + segment cut: the oracle's round trip starts from the reference's minimal line
    cuts = []
    for _ in range(30):
        line = rng.normal(size=6) * 4
        n = int(rng.integers(2, 9))
        cuts.append((line, np.ascontiguousarray(np.tile(line, (n, 1)) + rng.normal(scale=0.05, size=(n, 6)))))

    def minimal(L, pre, xs=None):
        getattr(L, pre + "minimal_from_line").argtypes = [C.c_void_p] * 2
        getattr(L, pre + "infinite_from_minimal").argtypes = [C.c_void_p] * 3
        getattr(L, pre + "segment_from_minimal").argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_void_p]
        p = orc._p
        out = np.zeros((len(cuts), 18))
        for k, (line, l3) in enumerate(cuts):
            getattr(L, pre + "minimal_from_line")(p(line), p(out[k, 0:6]))
            x = np.ascontiguousarray(out[k, 0:6] if xs is None else xs[k])
            getattr(L, pre + "infinite_from_minimal")(p(x), p(out[k, 6:9]), p(out[k, 9:12]))
            getattr(L, pre + "segment_from_minimal")(p(x), p(l3), len(l3), 1, p(out[k, 12:18]))
        return out

    def record():
        out = dict(minimal=minimal(ref.lib(), "ref_"))
        for no, (o2, l, sc, keep) in groups.items():
            out[f"aggregate_{no}"] = ref.aggregate_lines(o2, l, sc, no)[keep]
        return out
    r = _reference("aggregator_minimal", record)
    for no, (o2, l, sc, keep) in groups.items():
        a, b = orc.aggregate_lines(o2, l, sc, no)[keep], r[f"aggregate_{no}"]
        d = np.minimum(np.abs(a[:, :6] - b[:, :6]).max(1), np.abs(a[:, :6] - b[:, [3, 4, 5, 0, 1, 2]]).max(1))
        assert d.max() < 1e-8 and np.abs(a[:, 6] - b[:, 6]).max() == 0
    b = r["minimal"]
    a = minimal(orc.lib(), "orc_", xs=b[:, 0:6])
    for xa, xb in zip(a[:, 0:6], b[:, 0:6]):
        assert _close(xa, xb, 1e-9) or _close(np.concatenate([-xa[:4], xa[4:]]), xb, 1e-9)  # q == -q
    assert _close(a[:, 6:9], b[:, 6:9], 1e-12) and _close(a[:, 9:12], b[:, 9:12], 1e-10)
    assert _close(a[:, 12:18], b[:, 12:18], 1e-9)


def test_refinement_residual_functors():
    """a14/a15: the reference's GeometricRefinementFunctor / VPConstraintsFunctor (cost_functions.h), compiled and
    evaluated on forward-mode jets, against the restatement the LM oracle is built from: residuals AND the 6-column
    Jacobians, PINHOLE and SIMPLE_PINHOLE, unnormalised quaternions included."""
    rng = np.random.default_rng(306)
    L = orc.lib()
    L.orc_geometric_residual.argtypes = [C.c_void_p] * 5 + [C.c_double] + [C.c_void_p] * 2
    L.orc_vp_residual.argtypes = [C.c_void_p] * 6
    L.orc_minimal_from_line.argtypes = [C.c_void_p] * 2
    p = orc._p
    inputs = []
    for it in range(32):
        model = it & 1
        f = rng.uniform(300, 900)
        params = np.array([f, rng.uniform(300, 400), rng.uniform(200, 300)]) if model == 0 else \
            np.array([f, f * rng.uniform(0.9, 1.1), rng.uniform(300, 400), rng.uniform(200, 300)])
        kvec = np.array([params[0], params[0], params[1], params[2]]) if model == 0 else params.copy()
        q = rng.normal(size=4)
        q /= np.linalg.norm(q)
        q *= rng.choice([1.0, 1.0, 0.7, 1.3])     # ceres::QuaternionToRotation normalises: not assumed unit
        t = rng.normal(size=3) * 2
        line = rng.normal(size=6) * 3
        x = np.zeros(6)
        L.orc_minimal_from_line(p(line), p(x))
        x += rng.normal(scale=0.01, size=6)       # off the manifold too: the functors are ambient
        seg = rng.uniform(0, 700, 4)
        alpha = float(rng.choice([10.0, 0.0, 3.0]))
        vp = rng.normal(size=3)
        vp /= np.linalg.norm(vp)
        inputs.append((model, x, seg, params, kvec, q, t, alpha, vp))

    def record():
        R = ref.lib()
        out = np.zeros((len(inputs), 21))
        for k, (model, x, seg, params, kvec, q, t, alpha, vp) in enumerate(inputs):
            rb, jb, vb, vjb = np.zeros(2), np.zeros(12), np.zeros(1), np.zeros(6)
            R.ref_geometric_residual(model, p(x), p(seg), p(params), p(q), p(t), alpha, p(rb), p(jb))
            R.ref_vp_residual(model, p(x), p(vp), p(params), p(q), p(vb), p(vjb))
            out[k] = np.concatenate([rb, jb, vb, vjb])
        return dict(out=out)
    ref_out = _reference("residual_functors", record)["out"]
    worst = 0.0
    for it, ((model, x, seg, params, kvec, q, t, alpha, vp), o) in enumerate(zip(inputs, ref_out)):
        rb, jb, vb, vjb = o[0:2], o[2:14], o[14:15], o[15:21]
        ra, ja = np.zeros(2), np.zeros(12)
        L.orc_geometric_residual(p(x), p(seg), p(kvec), p(q), p(t), alpha, p(ra), p(ja))
        s = max(1.0, np.abs(rb).max())
        assert np.abs(ra - rb).max() <= 1e-9 * s, (it, ra, rb)
        sj = max(1.0, np.abs(jb).max())
        assert np.abs(ja - jb).max() <= 1e-8 * sj, (it, ja, jb)
        worst = max(worst, np.abs(ja - jb).max() / sj)
        va, vja = np.zeros(1), np.zeros(6)
        L.orc_vp_residual(p(x), p(vp), p(kvec), p(q), p(va), p(vja))
        assert abs(va[0] - vb[0]) <= 1e-10, (it, va, vb)
        assert np.abs(vja - vjb).max() <= 1e-8 * max(1.0, np.abs(vjb).max()), (it, vja, vjb)
    assert worst < 1e-8


def test_track_filters_and_remerge():
    from limap_b200.synth import make_track_lines, make_tracks
    ts = make_tracks(T=400, S=10, V=40, seed=305, noise_px=2.0)
    views, first = np.unique(ts.img_ids, return_index=True)
    remap = np.zeros(int(views.max()) + 1, np.int32)
    remap[views] = np.arange(len(views), dtype=np.int32)
    rng = np.random.default_rng(305)
    tl = ts.gt + rng.normal(scale=0.03, size=ts.gt.shape)
    a = (None, ts.kvec[first], ts.qvec[first], ts.tvec[first], ts.sup_off, remap[ts.img_ids], ts.segs, tl)
    kws = (dict(), dict(th_angular_2d=2.0, th_perp_2d=1.0, th_sv_angular_3d=60.0, th_overlap=0.9))
    lk = dict(score_th=0.5, th_angle=5.0, th_overlap=0.001, th_smartoverlap=0.1, th_smartangle=1.0, th_perp=1.0, th_innerseg=1.0)
    TL = make_track_lines(3000, dup_frac=0.4, seed=7, extent=8.0)
    acts = (np.ones(3000, np.uint8), (rng.random(3000) < 0.7).astype(np.uint8))

    def record():
        out = {f"flags_{k}": ref.track_support_flags(*a, **kw) for k, kw in enumerate(kws)}
        for k, act in enumerate(acts):
            out[f"group_{k}"], out[f"n_groups_{k}"] = ref.remerge_groups(TL, act, lk)
        return out
    r = _reference("track_filters_remerge", record)
    for k, kw in enumerate(kws):
        fa, fb = orc.track_support_flags(*a, **kw), r[f"flags_{k}"]
        assert np.array_equal(fa, fb) and 0 < (fa == 7).sum() < len(fa)
    for k, act in enumerate(acts):
        labels, ng, ne = orc.remerge_labels(TL, act, lk, threads=1)
        group, n_out = r[f"group_{k}"], int(r[f"n_groups_{k}"])
        # same partition: oracle labels <-> reference groups are in bijection
        pairs = set(zip(labels.tolist(), group.tolist()))
        assert len(pairs) == len(set(labels.tolist())) == len(set(group.tolist())) == ng == n_out
        assert ng < 3000


def test_golden_fixtures_consistent_with_recorded_reference_outputs():
    """Fixture consistency, no code under test: tests/golden/hotpath (frozen outputs of the oracle, the CUDA path's
    reference in test_golden_hotpath) against what the reference's compiled GlobalLineTriangulator computed on the same
    inputs when tests/golden/ref was recorded. It fails when a hot-path fixture is regenerated or edited into
    disagreement with the reference."""
    import test_golden_hotpath as g
    for name in g.TRI:
        z, cfg = g._load(name)
        img_ids = z["img_ids"]

        def record():
            t = ref.RefTri(cfg, threads=1)
            g._feed(t, z)
            return _tri_outputs(t, img_ids, 0)
        r = _reference(f"hotpath_{name}", record)
        assert np.array_equal(z["n_cand"], r["n_cand"])
        has = r["n_cand"] > 0
        assert np.array_equal(z["best_ng"][has], r["best_ng"][has])
        h = has[r["nodes"]]
        a, b = z["best_line"][r["nodes"]][h], r["best_line"][h]
        assert np.abs(a[:, :9] - b[:, :9]).max() <= 1e-4 and np.abs(a[:, 9] - b[:, 9]).max() <= 1e-6
        assert np.array_equal(z["edge_off"], r["edge_off"]) and np.array_equal(z["edges"], r["edges"])
        # the fixtures list tracks by sorted membership; the reference's come in graph order
        off = r["track_off"]
        members = [sorted(zip(r["track_img"][off[k]:off[k + 1]].tolist(), r["track_line_id"][off[k]:off[k + 1]].tolist()))
                   for k in range(len(off) - 1)]
        order = sorted(range(len(members)), key=lambda k: members[k])
        flat = np.asarray([m for k in order for m in members[k]], np.int32).reshape(-1, 2)
        assert np.array_equal(flat, z["track_members"])
        assert np.array_equal(np.concatenate([[0], np.cumsum([len(members[k]) for k in order])]), z["track_off"])
        pos = {k: j for j, k in enumerate(order)}
        for k in range(len(r["track_line"])):  # < 4 members: take-best ties (DESIGN.md §4)
            if len(members[k]) >= 4:
                a, b = z["track_line"][pos[k]], r["track_line"][k]
                assert min(np.abs(a[:6] - b[:6]).max(), np.abs(a[:6] - b[[3, 4, 5, 0, 1, 2]]).max()) <= 1e-4


def test_sfm_model_neighbour_ranking_and_ranges():
    """f4: the reference's compiled pointsfm/sfm_model.cc (ranking loops, IoU / Dice formulas, sorts, ComputeRanges float
    arithmetic; COLMAP's mvs::Model statistics restated in oracle/ref_shim) against the oracle restatement the CUDA path
    is tested with. The reference orders equal scores with an UNSTABLE sort, the restatement keeps ascending image index:
    lists are compared exactly where the scores are distinct and by score sequence where they tie."""
    from limap_b200.base import CameraPose
    from limap_b200.synth import make_scene, make_sfm_points
    for seed, V, n_pts in ((71, 30, 4000), (72, 12, 300)):
        sc = make_scene(V=V, L=10, N=3, K=1, seed=seed)
        _, xyz, off, img = make_sfm_points(sc, n_points=n_pts, seed=seed)
        R = np.stack([CameraPose(sc.qvec[v], sc.tvec[v]).R() for v in range(V)])
        T = sc.tvec
        centres = ref.colmap_float_centres(R, T)
        xyz32 = xyz.astype(np.float32).astype(np.float64)  # Model::Point keeps float coordinates
        rankings = [(mode, n_nb, ang) for mode in (0, 1, 2) for n_nb, ang in ((8, 1.0), (100, 0.5), (3, 6.0))]
        quantiles = ((0.05, 0.95, 1.25), (0.0, 0.999, 0.5), (0.25, 0.5, 2.0))

        def record():
            out = {}
            for mode, n_nb, ang in rankings:
                out[f"rank_{mode}_{n_nb}"], out[f"count_{mode}_{n_nb}"] = ref.sfm_rank_neighbors(
                    R, T, xyz, off, img, n_nb, min_triangulation_angle=ang, mode=mode)
            for k, q in enumerate(quantiles):
                out[f"lo_{k}"], out[f"hi_{k}"] = ref.sfm_robust_ranges(xyz, *q)
            return out
        r = _reference(f"sfm_model_{seed}", record)
        # scores per (i, j) for the tie analysis
        shared = np.zeros((V, V), np.int64)
        npts = np.bincount(img, minlength=V)
        for p in range(len(off) - 1):
            t = img[off[p]:off[p + 1]]
            shared[np.ix_(t, t)] += 1
        np.fill_diagonal(shared, 0)
        for mode in (0, 1, 2):
            union = npts[:, None] + npts[None, :] - shared
            score = (shared / np.maximum(union, 1), 2 * shared / np.maximum(union + shared, 1), shared.astype(float))[mode]
            for n_nb, ang in ((8, 1.0), (100, 0.5), (3, 6.0)):
                a, ca = orc.rank_neighbors(centres, xyz32, off, img, n_nb, min_triangulation_angle=ang, mode=mode)
                b, cb = r[f"rank_{mode}_{n_nb}"], r[f"count_{mode}_{n_nb}"]
                assert np.array_equal(ca, cb), (seed, mode, n_nb, ang)
                n_exact = 0
                for i in range(V):
                    la, lb = a[i, :ca[i]], b[i, :cb[i]]
                    sa, sb = score[i, la], score[i, lb]
                    assert np.array_equal(sa, sb), (seed, mode, n_nb, ang, i)  # same scores in the same order
                    row = score[i, shared[i] > 0]
                    if all((row == v).sum() == 1 for v in sa):  # no listed score ties with any other co-visible image
                        assert np.array_equal(la, lb), (seed, mode, n_nb, ang, i)
                        n_exact += 1
                assert n_exact > 0 or mode == 2
        for k, q in enumerate(quantiles):
            lo_a, hi_a = orc.robust_ranges(xyz, *q)
            assert np.array_equal(lo_a, r[f"lo_{k}"]) and np.array_equal(hi_a, r[f"hi_{k}"]), q  # float arithmetic, bit for bit


def test_jlinkage_wrapper_filtering_renumbering_and_vp_fit():
    """a18: limap's own J-Linkage wrapper (vplib/JLinkage/JLinkage.cc + base_vp_detector.cc: min_length filter, the 2 x
    max(min_num_supports, 10) guard, cluster filtering with count_valid_supports_2d, label renumbering, VP = last right
    singular vector of the stacked line coordinates) compiled unchanged, over a JLinkage-library shim that forwards the
    sampling / clustering to the restated core -- against the restatement of the same wrapper in oracle/orc_vp.h.
    (The JLinkage library itself is an absent submodule: its core stays restated, DESIGN.md 6.)"""
    from limap_b200.synth import make_vp_images
    imgs = make_vp_images(6, 120, seed=81) + make_vp_images(2, 25, seed=82) + [np.zeros((0, 4))]
    imgs = [np.ascontiguousarray(segs, np.float64).reshape(-1, 4) for segs in imgs]
    kws = (dict(), dict(min_length=20.0, min_num_supports=8, th_perp_supports=1.0), dict(inlier_threshold=2.5))

    def record():
        out = {}
        for idx, segs in enumerate(imgs):
            for k, kw in enumerate(kws):
                out[f"labels_{idx}_{k}"], out[f"vps_{idx}_{k}"] = ref.vp_associate(segs, seed=7, image_index=idx, **kw)
        return out
    r = _reference("jlinkage_wrapper", record)
    n_vp_total = 0
    for idx, segs in enumerate(imgs):
        for k, kw in enumerate(kws):
            la, va = r[f"labels_{idx}_{k}"], r[f"vps_{idx}_{k}"]
            off = np.array([0, len(segs)], np.int64)
            lb, _, vb = orc.detect_vps(off, segs, n_models=5000, seed=7, image_index=[idx], threads=1, **kw)
            assert np.array_equal(la, lb), (idx, kw)
            assert len(va) == len(vb)
            for a, b in zip(va, vb):
                assert min(np.abs(a - b).max(), np.abs(a + b).max()) < 1e-7, (idx, kw, a, b)  # sign of a singular vector
            n_vp_total += len(va)
    assert n_vp_total >= 10


def test_linetrack_file_format_and_line_weights(tmp_path):
    """a19: LineTrack::Write / LineTrack::Read of the reference's compiled base/linetrack.cc against the Python mirror
    (limap_b200.base.LineTrack): the mirror's writer reproduces the reference's bytes, each side reads the other's file;
    ComputeLineWeights (the loss weight of a supporting line in the refinement) = length / 30."""
    import limap.base as base
    rng = np.random.default_rng(91)
    p = orc._p
    cases = []
    for case in range(6):
        n = int(rng.integers(1, 9))
        line = rng.normal(size=6) * 3
        if case == 4:
            line[1] = np.nan  # written as 0 (linetrack.cc:137-152)
        img = rng.integers(0, 5, n).astype(np.int32)
        lid = rng.integers(0, 400, n).astype(np.int32)
        node = rng.integers(0, 10 ** 6, n).astype(np.int32)
        score = rng.uniform(0, 5, n)
        l2d = rng.uniform(0, 800, (n, 4))
        l3d = rng.normal(size=(n, 6)) * 2
        aux = case != 5  # case 5: a track without node ids / scores / 3D lines
        t = base.LineTrack()
        t.line = base.Line3d(line[:3], line[3:])
        t.image_id_list, t.line_id_list = img.tolist(), lid.tolist()
        t.line2d_list = [base.Line2d(r[:2], r[2:]) for r in l2d]
        if aux:
            t.node_id_list, t.score_list = node.tolist(), score.tolist()
            t.line3d_list = [base.Line3d(r[:3], r[3:]) for r in l3d]
        f_py = str(tmp_path / f"py_{case}.txt")
        t.Write(f_py)
        cases.append((n, line, img, lid, node, score, l2d, l3d, aux, f_py))
    segs = rng.uniform(0, 800, (200, 4))

    def record():
        L, out = ref.lib(), {}
        for case, (n, line, img, lid, node, score, l2d, l3d, aux, f_py) in enumerate(cases):
            f_ref = str(tmp_path / f"ref_{case}.txt").encode()
            L.ref_linetrack_write(f_ref, p(line), n, p(img), p(lid), p(node) if aux else None, p(score) if aux else None,
                                  p(l2d), p(l3d) if aux else None)
            with open(f_ref.decode(), "rb") as f:
                out[f"file_{case}"] = np.frombuffer(f.read(), np.uint8)
            # the reference reads the mirror's file
            o = dict(line=np.zeros(6), img=np.zeros(n, np.int32), lid=np.zeros(n, np.int32), node=np.zeros(n, np.int32),
                     score=np.zeros(n), l2d=np.zeros((n, 4)), l3d=np.zeros((n, 6)), n_images=np.zeros(1, np.int32))
            out[f"read_count_{case}"] = L.ref_linetrack_read(f_py.encode(), n, *[p(v) for v in o.values()])
            out.update({f"read_{k}_{case}": v for k, v in o.items()})
        w = np.zeros(200)
        L.ref_line_weights(200, p(segs), p(w))
        out["weights"] = w
        return out
    r = _reference("linetrack", record)
    for case, (n, line, img, lid, node, score, l2d, l3d, aux, f_py) in enumerate(cases):
        f_ref = tmp_path / f"ref_{case}.txt"
        f_ref.write_bytes(r[f"file_{case}"].tobytes())
        with open(f_py, "rb") as f:
            assert f.read() == f_ref.read_bytes(), case  # byte for byte
        # the mirror reads the reference's file
        t2 = base.LineTrack()
        t2.Read(str(f_ref))
        assert t2.image_id_list == img.tolist() and t2.line_id_list == lid.tolist() and t2.count_images() == len(set(img))
        assert np.allclose([np.concatenate([l.start, l.end]) for l in t2.line2d_list], l2d, atol=1e-9)
        if aux:
            assert t2.node_id_list == node.tolist() and np.allclose(t2.score_list, score, atol=1e-9)
            assert np.allclose([np.concatenate([l.start, l.end]) for l in t2.line3d_list], l3d, atol=1e-9)
        # the reference reads the mirror's file
        o = lambda k: r[f"read_{k}_{case}"]
        assert int(r[f"read_count_{case}"]) == n and np.array_equal(o("img"), img) and np.array_equal(o("lid"), lid)
        assert o("n_images")[0] == len(set(img))
        assert np.allclose(o("line"), np.nan_to_num(line), atol=1e-9) and np.allclose(o("l2d"), l2d, atol=1e-9)
        if aux:
            assert np.array_equal(o("node"), node) and np.allclose(o("score"), score, atol=1e-9)
            assert np.allclose(o("l3d"), l3d, atol=1e-9)
    dx, dy = segs[:, 2] - segs[:, 0], segs[:, 3] - segs[:, 1]
    assert np.allclose(r["weights"], np.sqrt(dx * dx + dy * dy) / 30.0, rtol=1e-15, atol=0)


def test_python_value_types_against_compiled_reference():
    """a1 / a19: the Python value types of the mirror (limap_b200.base: Camera, CameraPose, CameraView, Line2d, Line3d) --
    the objects a runner handles -- against the reference's compiled base/{camera,pose,camera_view,linebase}.cc:
    projection, ray_direction, Line2d length / direction, Line3d sensitivity and uncertainty."""
    import limap.base as base
    rng = np.random.default_rng(92)
    p = orc._p
    inputs = []
    for it in range(80):
        model = it & 1
        f = rng.uniform(300, 900)
        fy = f if model == 0 else f * rng.uniform(0.9, 1.1)
        cx, cy = rng.uniform(300, 400), rng.uniform(200, 300)
        q = rng.normal(size=4)
        q /= np.linalg.norm(q)
        t = rng.normal(size=3) * 3
        cam_arr = np.array([model, f, fy, cx, cy, *q, *t])
        cam = base.Camera("SIMPLE_PINHOLE", [f, cx, cy], 0, (600, 800)) if model == 0 else \
            base.Camera("PINHOLE", [f, fy, cx, cy], 0, (600, 800))
        view = base.CameraView(cam, base.CameraPose(q, t))
        X = rng.normal(size=3) * 2 + view.pose.center() + view.R().T @ np.array([0, 0, 6.0])
        px = rng.uniform(0, 700, 2)
        seg = rng.uniform(0, 700, 4)
        Y = rng.normal(size=3) * 2 + view.pose.center() + view.R().T @ np.array([0, 0, 7.0])
        l3_arr = np.array([*X, *Y, view.pose.projdepth(X), view.pose.projdepth(Y), 0.1])
        inputs.append((cam_arr, view, X, px, seg, Y, l3_arr))

    def record():
        L = ref.lib()
        out = np.zeros((len(inputs), 10))
        for k, (cam_arr, view, X, px, seg, Y, l3_arr) in enumerate(inputs):
            L.ref_project_point(p(cam_arr), p(X), p(out[k, 0:2]))
            r = np.zeros(3)
            L.ref_ray_direction(p(cam_arr), p(px), p(r))
            out[k, 2:5] = r
            out[k, 5] = L.ref_line2d_length(p(seg))
            d = np.zeros(2)
            L.ref_line2d_direction(p(seg), p(d))
            out[k, 6:8] = d
            out[k, 8] = L.ref_line3d_sensitivity(p(l3_arr), p(cam_arr))
            out[k, 9] = L.ref_line3d_uncertainty(p(l3_arr), p(cam_arr), 5.0)
        return dict(out=out)
    r = _reference("value_types", record)["out"]
    for it, ((cam_arr, view, X, px, seg, Y, l3_arr), o) in enumerate(zip(inputs, r)):
        b = o[0:2]
        a = np.asarray(view.projection(X))
        assert np.abs(a - b).max() <= 1e-9 * max(1.0, np.abs(b).max()), (it, a, b)
        assert np.abs(np.asarray(view.ray_direction(px)) - o[2:5]).max() <= 1e-12
        l2 = base.Line2d(seg[:2], seg[2:])
        assert abs(l2.length() - o[5]) <= 1e-12 and np.abs(np.asarray(l2.direction()) - o[6:8]).max() <= 1e-12
        l3 = base.Line3d(X, Y, 1.0, float(l3_arr[6]), float(l3_arr[7]), 0.1)
        assert abs(l3.sensitivity(view) - o[8]) <= 1e-7
        assert abs(l3.computeUncertainty(view, 5.0) - o[9]) <= 1e-10 * max(1.0, abs(l3_arr[6]))


def _flatten_tracks(tracks, view_of):
    off, tl, act, view, lid, node, score, l2d, l3d = [0], [], [], [], [], [], [], [], []
    l9 = lambda l: [*l.start, *l.end, l.depths[0], l.depths[1], l.uncertainty]
    for t in tracks:
        tl.append(l9(t.line))
        act.append(1 if t.active else 0)
        for k in range(t.count_lines()):
            view.append(view_of[int(t.image_id_list[k])])
            lid.append(int(t.line_id_list[k]))
            node.append(int(t.node_id_list[k]))
            score.append(float(t.score_list[k]))
            l2d.append([*t.line2d_list[k].start, *t.line2d_list[k].end])
            l3d.append(l9(t.line3d_list[k]))
        off.append(len(view))
    f = lambda a, dt, shp: np.ascontiguousarray(np.asarray(a, dt).reshape(shp))
    return (f(off, np.int64, -1), f(tl, np.float64, (-1, 9)), f(act, np.uint8, -1), f(view, np.int32, -1), f(lid, np.int32, -1),
            f(node, np.int32, -1), f(score, np.float64, -1), f(l2d, np.float64, (-1, 4)), f(l3d, np.float64, (-1, 9)))


def _ref_track_filter(op, a, b, n, lk, cams, flat):
    """One track-level operator of the reference's compiled merging code on flattened tracks. Returned: track offsets,
    track lines, active flags and, per output support, the index of the input support it is (supports are carried over
    unchanged: checked here field by field)."""
    L = ref.lib()
    p = orc._p
    off, tl, act, view, lid, node, score, l2d, l3d = flat
    T, S = len(off) - 1, len(view)
    o = (np.zeros(T + 1, np.int64), np.zeros((max(T, 1), 9)), np.zeros(max(T, 1), np.uint8), np.zeros(max(S, 1), np.int32),
         np.zeros(max(S, 1), np.int32), np.zeros(max(S, 1), np.int32), np.zeros(max(S, 1)), np.zeros((max(S, 1), 4)),
         np.zeros((max(S, 1), 9)))
    model_ids, kvec, qvec, tvec = cams
    cfg = ref.linker_cfg(lk or {})
    To = L.ref_track_filter(op, float(a), float(b), int(n), C.byref(cfg), len(kvec), p(model_ids), p(kvec), p(qvec), p(tvec), T,
                            p(off), p(tl), p(act), p(view), p(lid), p(node), p(score), p(l2d), p(l3d), *[p(x) for x in o])
    S_o = int(o[0][To])
    key = {(int(v), int(l), int(d)): k for k, (v, l, d) in enumerate(zip(view, lid, node))}
    assert len(key) == S
    src = np.array([key[(int(v), int(l), int(d))] for v, l, d in zip(o[3][:S_o], o[4][:S_o], o[5][:S_o])], np.int64)
    assert np.array_equal(o[6][:S_o], score[src]) and np.array_equal(o[7][:S_o], l2d[src]) and np.array_equal(o[8][:S_o], l3d[src])
    return dict(track_off=o[0][:To + 1], track_line=o[1][:To, :6], active=o[2][:To], support=src)


def test_track_level_filters_and_remerge_against_compiled_reference(monkeypatch):
    """f1 at track level: the mirror's post-triangulation operators (limap_b200.merging: list surgery in Python on top of the
    engine's per-support predicates, here served by the oracle stand-in so that the test runs without a GPU) against the
    reference's compiled FilterSupportingLines / FilterTracksBySensitivity / FilterTracksByOverlap / iterated
    RemergeLineTracks, on the tracks of a triangulated scene: same tracks in the same order, same supports, same lines."""
    import limap.base as base
    import limap.merging as merging
    import limap.triangulation as triangulation
    from limap_b200.config import DEFAULT_YAML_TRIANGULATION
    from limap_b200.synth import make_scene
    from runner_utils import imagecols_of, install_oracle_backend
    install_oracle_backend(monkeypatch)
    sc = make_scene(V=10, L=120, N=5, K=4, seed=93, noise_px=1.0, camera_mix=True)
    imagecols = imagecols_of(sc)
    tri = triangulation.GlobalLineTriangulator(dict(DEFAULT_YAML_TRIANGULATION))
    tri.SetRanges(sc.ranges)
    tri.Init({int(i): [base.Line2d(s[:2], s[2:]) for s in sc.lines_of(v)] for v, i in enumerate(sc.img_ids)}, imagecols)
    for i in sc.img_ids:
        tri.TriangulateImage(int(i), sc.matches[int(i)])
    tracks = tri.ComputeLineTracks()
    assert len(tracks) > 30
    view_of = {int(i): v for v, i in enumerate(sc.img_ids)}
    cams = (np.ascontiguousarray(sc.model_ids, np.int32), sc.kvec, sc.qvec, sc.tvec)

    def same(py_tracks, tracks_in, op, a, b, n, lk, tag):
        flat_in = _flatten_tracks(tracks_in, view_of)
        r = _reference(f"track_level_{tag}", lambda: _ref_track_filter(op, a, b, n, lk, cams, flat_in))
        got = _flatten_tracks(py_tracks, view_of)
        src = r["support"]
        assert np.array_equal(got[0], r["track_off"]), tag                   # track boundaries
        for k in (3, 4, 5):                                                  # views, line ids, node ids in order
            assert np.array_equal(got[k], flat_in[k][src]), (tag, k)
        assert np.array_equal(got[2], r["active"]), tag                      # active flags
        assert np.allclose(got[6], flat_in[6][src], atol=1e-12) and np.allclose(got[7], flat_in[7][src], atol=1e-12)
        tl = r["track_line"]
        d = np.minimum(np.abs(got[1][:, :6] - tl).max(1, initial=0), np.abs(got[1][:, :6] - tl[:, [3, 4, 5, 0, 1, 2]]).max(1, initial=0))
        assert d.max(initial=0) < 1e-8, (tag, d.max())
        return len(py_tracks)

    n0 = len(tracks)
    t1 = merging.filter_tracks_by_reprojection(tracks, imagecols, 4.0, 2.0, num_outliers=0)
    n1 = same(t1, tracks, 0, 4.0, 2.0, 0, None, "reprojection")
    lk = dict(score_th=0.5, th_angle=8.0, th_overlap=0.01, th_smartoverlap=0.1, th_smartangle=1.0, th_perp=1.0, th_innerseg=1.0)
    t2 = merging.remerge(base.LineLinker3d(lk), t1, num_outliers=0)
    n2 = same(t2, t1, 3, 0, 0, 0, lk, "remerge")
    t3 = merging.filter_tracks_by_sensitivity(t2, imagecols, 75.0, 4)
    n3 = same(t3, t2, 1, 75.0, 0, 4, None, "sensitivity")
    t4 = merging.filter_tracks_by_overlap(t3, imagecols, 0.5, 4)
    n4 = same(t4, t3, 2, 0.5, 0, 4, None, "overlap")
    assert n0 >= n1 >= n2 >= n3 >= n4 > 5 and n4 < n0


def test_camera_set_max_image_dim_rounding():
    """Camera::set_max_image_dim (the runner's max_image_dim): the new size is C round() of ratio * size (halves away from
    zero, not to even), the intrinsics follow colmap::Camera::Rescale."""
    import limap.base as base
    rng = np.random.default_rng(94)
    cases = [(801, 1602, 801), (600, 800, 400), (1000, 3, 500)]  # (h, w, val): the first has ratio * h == 400.5 exactly
    cases += [(int(rng.integers(100, 3000)), int(rng.integers(100, 3000)), int(rng.integers(50, 3500))) for _ in range(100)]
    params = {0: [612.3, 400.5, 299.25], 1: [612.3, 640.7, 400.5, 299.25]}

    def record():
        L = ref.lib()
        L.ref_camera_set_max_image_dim.argtypes = [C.c_int, C.c_void_p, C.c_void_p, C.c_int]
        out = dict(hw=np.zeros((len(cases), 2, 2), np.int32), params=np.zeros((len(cases), 2, 4)))
        for k, (h, w, val) in enumerate(cases):
            for model in (0, 1):
                pr = np.array(params[model] + [0.0] * (4 - len(params[model])))
                hw = np.array([h, w], np.int32)
                L.ref_camera_set_max_image_dim(model, orc._p(pr), orc._p(hw), val)
                out["hw"][k, model], out["params"][k, model] = hw, pr
        return out
    r = _reference("camera_set_max_image_dim", record)
    n_half = 0
    for k, (h, w, val) in enumerate(cases):
        for model in (0, 1):
            cam = base.Camera("SIMPLE_PINHOLE" if model == 0 else "PINHOLE", list(params[model]), 0, (h, w))
            cam.set_max_image_dim(val)
            hw, pr = r["hw"][k, model], r["params"][k, model]
            assert (cam.h(), cam.w()) == (int(hw[0]), int(hw[1])), (h, w, val)
            assert np.allclose(cam.params, pr[:len(params[model])], rtol=1e-15, atol=0), (h, w, val)
        ratio = val / max(h, w)
        n_half += ratio < 1 and (abs(ratio * h % 1 - 0.5) < 1e-12 or abs(ratio * w % 1 - 0.5) < 1e-12)
    assert n_half >= 1
