"""Row preparation by the per-view stable counting sort (row_count / row_scan / row_scatter, the default) against the
radix-sort path (expand_rows -> stable radix sort by node id -> node_offsets, LIMAP_B200_ROW_SORT=cub). A stable sort
has exactly one result, so every output must be bit-identical: node records (floats compared by their bits), valid-edge
offsets and edges, debug_mode candidate lists, and the run statistics that depend on the rows."""
import numpy as np
import pytest

from limap_b200._cabi import LimapB200Error
from limap_b200.config import DEFAULT_YAML_TRIANGULATION
from limap_b200.synth import CONFIGS, concat_scenes, make_scene

from test_tri_parity_gpu import _fake_vpresults

pytestmark = pytest.mark.gpu

ROW_SORT_MAX_LINES = 4096  # kRowSortMaxLines in tri_kernels.cuh: views with more lines keep the radix-sort path


def _cfg(**kw):
    c = dict(DEFAULT_YAML_TRIANGULATION)
    c.update(kw)
    return c


def _engine(sc, cfg, vpresults=None, shard=None, groups=None, bulk=False):
    from limap_b200.engine import TriEngine
    eng = TriEngine(cfg)
    eng.upload(sc)
    eng.set_ranges(*sc.ranges)
    if vpresults is not None:
        eng.set_vps(vpresults, sc.img_ids, sc.line_off)
    if bulk:
        eng.add_matches_bulk(*sc.bulk_matches())
    else:
        for i in sc.img_ids:
            eng.add_image_matches(int(i), *sc.flat_matches(int(i)))
    if shard is not None:
        eng.set_shard(*shard)
    if groups is not None:
        eng.set_pipeline_groups(groups)
    return eng


def _set_path(monkeypatch, cub):
    if cub:
        monkeypatch.setenv("LIMAP_B200_ROW_SORT", "cub")
    else:
        monkeypatch.delenv("LIMAP_B200_ROW_SORT", raising=False)


def _outputs(eng, cub, monkeypatch, debug_nodes=()):
    _set_path(monkeypatch, cub)
    st = eng.run()
    nodes = eng.get_nodes()
    off, edges = eng.get_all_valid_edges()
    cands = [eng.get_cands_node(int(i), int(l)) for i, l in debug_nodes]
    monkeypatch.delenv("LIMAP_B200_ROW_SORT", raising=False)
    return dict(st=st, nodes=nodes, off=off, edges=edges, cands=cands)


def _bits(x):
    return np.ascontiguousarray(x).view(np.uint8)


def _assert_identical(a, b):
    na, nb = a["nodes"], b["nodes"]
    assert na.dtype == nb.dtype and na.shape == nb.shape
    for f in na.dtype.names:
        assert np.array_equal(_bits(na[f]), _bits(nb[f])), f
    assert np.array_equal(a["off"], b["off"])
    assert np.array_equal(a["edges"], b["edges"])
    assert len(a["cands"]) == len(b["cands"])
    for (la, ga), (lb, gb) in zip(a["cands"], b["cands"]):
        assert np.array_equal(ga, gb)
        assert np.array_equal(_bits(la), _bits(lb))
    for k in ("n_rows", "n_candidates", "n_valid_edges", "n_pairs_gated", "n_pairs_exact", "max_rows_per_node"):
        assert a["st"][k] == b["st"][k], k


def _all_nodes(sc):
    return [(int(i), l) for v, i in enumerate(sc.img_ids) for l in range(int(sc.line_off[v + 1] - sc.line_off[v]))]


def _check(eng, monkeypatch, debug_nodes=()):
    new = _outputs(eng, False, monkeypatch, debug_nodes)
    _assert_identical(new, _outputs(eng, True, monkeypatch, debug_nodes))
    assert new["st"]["n_candidates"] > 0
    return new


@pytest.fixture(scope="module")
def hypersim100():
    return make_scene(**CONFIGS["hypersim100"])


@pytest.mark.parametrize("groups", [1, 8])
def test_hypersim100_counting_sort_equals_radix_sort(hypersim100, groups, monkeypatch):
    eng = _engine(hypersim100, _cfg(), groups=groups, bulk=True)
    new = _check(eng, monkeypatch)
    assert new["st"]["n_valid_edges"] > 0


def test_shuffled_rows(monkeypatch):
    sc = make_scene(V=10, L=250, N=6, K=8, seed=51, shuffle_rows=True)
    _check(_engine(sc, _cfg(debug_mode=True)), monkeypatch, _all_nodes(sc))


def test_view_shard(monkeypatch):
    sc = make_scene(V=12, L=300, N=8, K=10, seed=31)
    _check(_engine(sc, _cfg(), shard=(3, 9)), monkeypatch)


def test_vp_proposals(monkeypatch):
    sc = make_scene(V=6, L=60, N=4, K=3, seed=21)
    eng = _engine(sc, _cfg(use_vp=True, debug_mode=True), vpresults=_fake_vpresults(sc, 5))
    new = _check(eng, monkeypatch, _all_nodes(sc))
    assert sum(len(c[0]) for c in new["cands"]) == new["st"]["n_candidates"]


def test_images_and_lines_without_matches(monkeypatch):
    sc = make_scene(V=12, L=400, N=8, K=8, seed=53)  # about 2e5 rows: three pipeline groups
    rng = np.random.default_rng(6)
    ids = list(sc.img_ids)
    for v, i in enumerate(ids):
        m = sc.matches[int(i)]
        L = int(sc.line_off[v + 1] - sc.line_off[v])
        empty = rng.random(L) < 0.3  # lines without any match row
        for g in list(m.keys()):
            keep = np.zeros(len(m[g]), bool) if v in (0, 4) else ~empty[m[g][:, 0]]  # images 0 and 4: no matches
            m[g] = np.ascontiguousarray(m[g][keep])
    for groups in (1, 3):
        eng = _engine(sc, _cfg(debug_mode=True), groups=groups)
        new = _check(eng, monkeypatch, _all_nodes(sc))
        nc = new["nodes"]["n_cand"]
        assert (nc[sc.line_off[0]:sc.line_off[1]] == 0).all() and (nc[sc.line_off[4]:sc.line_off[5]] == 0).all()


@pytest.mark.parametrize("big_first", [True, False])
def test_view_above_histogram_bound_next_to_counting_sort(big_first, monkeypatch):
    small = make_scene(V=5, L=200, N=3, K=4, seed=55)
    big = make_scene(V=3, L=ROW_SORT_MAX_LINES + 100, N=2, K=2, seed=56)
    small2 = make_scene(V=4, L=120, N=3, K=3, seed=57)
    sc = concat_scenes([big, small, small2] if big_first else [small, big, small2])
    lines = np.diff(sc.line_off)
    assert (lines > ROW_SORT_MAX_LINES).any() and (lines <= ROW_SORT_MAX_LINES).any()
    debug = [n for n in _all_nodes(sc) if n[1] % 7 == 0]
    _check(_engine(sc, _cfg(debug_mode=True)), monkeypatch, debug)


@pytest.mark.parametrize("which", ["line", "neighbour_line"])
def test_out_of_range_line_id_raises_on_both_paths(which, monkeypatch):
    sc = make_scene(V=6, L=80, N=3, K=3, seed=58)
    i = int(sc.img_ids[2])
    g = next(iter(sc.matches[i]))
    rows = sc.matches[i][g].copy()
    rows[len(rows) // 2, 0 if which == "line" else 1] = 10_000
    sc.matches[i][g] = rows
    msgs = []
    for cub in (False, True):
        eng = _engine(sc, _cfg())
        _set_path(monkeypatch, cub)
        with pytest.raises(LimapB200Error, match="IndexError") as ei:
            eng.run()
        msgs.append(str(ei.value))
    monkeypatch.delenv("LIMAP_B200_ROW_SORT", raising=False)
    assert msgs[0] == msgs[1]


def test_two_consecutive_runs_on_one_engine(monkeypatch):
    sc = make_scene(V=10, L=200, N=6, K=6, seed=59)
    eng = _engine(sc, _cfg(debug_mode=True), groups=2)
    nodes = _all_nodes(sc)
    first = _outputs(eng, False, monkeypatch, nodes)
    second = _outputs(eng, False, monkeypatch, nodes)
    ref = _outputs(_engine(sc, _cfg(debug_mode=True), groups=2), True, monkeypatch, nodes)
    _assert_identical(first, ref)
    _assert_identical(second, ref)
