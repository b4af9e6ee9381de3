"""The split form of the fast triangulation path (tri_gen_kernel + tri_score_kernel) against the fused tri_node_kernel
(LIMAP_B200_TRI_FUSED=1). Candidate counts, best-candidate indices, valid connections and debug_mode candidate lists
must be identical. The fp64 values (3D endpoints, depths, uncertainty, scores) agree to the last bits only: the two
kernels evaluate the same expressions, but the compiler contracts multiply-adds into FMAs differently in each, so they
are compared at a relative tolerance of 1e-9 -- five orders below the 1e-4 parity tolerance against the oracle."""
import numpy as np
import pytest

from limap_b200.config import DEFAULT_YAML_TRIANGULATION
from limap_b200.synth import CONFIGS, make_scene

from test_tri_parity_gpu import _fake_vpresults

pytestmark = pytest.mark.gpu


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


def _outputs(eng, fused, monkeypatch, debug_nodes=()):
    if fused:
        monkeypatch.setenv("LIMAP_B200_TRI_FUSED", "1")
    else:
        monkeypatch.delenv("LIMAP_B200_TRI_FUSED", raising=False)
    st = eng.run()
    nodes = eng.get_nodes()
    off, edges = eng.get_all_valid_edges()
    cands = [eng.get_cands_node(int(i), int(l)) for i, l in debug_nodes]
    monkeypatch.delenv("LIMAP_B200_TRI_FUSED", raising=False)
    return dict(st=st, nodes=nodes, off=off, edges=edges, cands=cands)


FP_RTOL = 1e-9


def _close(x, y):
    assert x.shape == y.shape
    np.testing.assert_allclose(x, y, rtol=FP_RTOL, atol=FP_RTOL)


def _assert_same(a, b):
    na, nb = a["nodes"], b["nodes"]
    for f in na.dtype.names:
        if np.issubdtype(na[f].dtype, np.floating):
            _close(na[f], nb[f])
        else:
            assert np.array_equal(na[f], nb[f]), f
    assert np.array_equal(a["off"], b["off"])
    assert np.array_equal(a["edges"], b["edges"])
    assert len(a["cands"]) == len(b["cands"])
    for (la, ga), (lb, gb) in zip(a["cands"], b["cands"]):
        assert np.array_equal(ga, gb)
        _close(la, lb)
    for k in ("n_candidates", "n_valid_edges", "n_pairs_gated", "n_pairs_exact"):
        assert a["st"][k] == b["st"][k], k


def _all_nodes(sc):
    return [(int(i), l) for v, i in enumerate(sc.img_ids) for l in range(int(sc.line_off[v + 1] - sc.line_off[v]))]


@pytest.fixture(scope="module")
def hypersim100():
    return make_scene(**CONFIGS["hypersim100"])


@pytest.mark.parametrize("groups", [1, 4, 8])
def test_hypersim100_split_equals_fused(hypersim100, groups, monkeypatch):
    eng = _engine(hypersim100, _cfg(), groups=groups, bulk=True)
    fused = _outputs(eng, True, monkeypatch)
    split = _outputs(eng, False, monkeypatch)
    _assert_same(split, fused)
    assert split["st"]["n_candidates"] > 0 and split["st"]["n_valid_edges"] > 0


def test_shard_split_equals_fused(monkeypatch):
    sc = make_scene(V=12, L=300, N=8, K=10, seed=31)
    eng = _engine(sc, _cfg(), shard=(3, 9))
    _assert_same(_outputs(eng, False, monkeypatch), _outputs(eng, True, monkeypatch))


def test_vp_proposals_split_equals_fused(monkeypatch):
    sc = make_scene(V=6, L=60, N=4, K=3, seed=21)
    eng = _engine(sc, _cfg(use_vp=True, debug_mode=True), vpresults=_fake_vpresults(sc, 5))
    nodes = _all_nodes(sc)
    split = _outputs(eng, False, monkeypatch, nodes)
    _assert_same(split, _outputs(eng, True, monkeypatch, nodes))
    assert sum(len(c[0]) for c in split["cands"]) == split["st"]["n_candidates"] > 0


def test_empty_and_ragged_nodes_split_equals_fused(monkeypatch):
    sc = make_scene(V=8, L=120, N=5, K=6, seed=33)
    rng = np.random.default_rng(4)
    for i, m in sc.matches.items():
        L = int(sc.line_off[list(sc.img_ids).index(i) + 1] - sc.line_off[list(sc.img_ids).index(i)])
        empty = rng.random(L) < 0.3  # lines without any match row
        for g in list(m.keys()):
            keep = ~empty[m[g][:, 0]] & (rng.random(len(m[g])) < rng.random())  # ragged row counts
            m[g] = np.ascontiguousarray(m[g][keep])
    eng = _engine(sc, _cfg(debug_mode=True))
    nodes = _all_nodes(sc)
    split = _outputs(eng, False, monkeypatch, nodes)
    _assert_same(split, _outputs(eng, True, monkeypatch, nodes))
    nc = split["nodes"]["n_cand"]
    assert (nc == 0).any() and len(np.unique(nc)) > 5


def test_candidate_capacity_retry(monkeypatch):
    # a low-candidate scene sizes the scorer's staging area at 32; the next scene has more candidates per node, so its
    # first pass overflows and the run repeats once with the exact size
    monkeypatch.delenv("LIMAP_B200_TRI_FUSED", raising=False)
    small = make_scene(V=6, L=60, N=3, K=2, seed=41)
    big = make_scene(V=8, L=120, N=8, K=10, seed=42)
    eng = _engine(small, _cfg())
    st = eng.run()
    assert 0 < st["n_candidates"]
    eng.clear()
    eng.upload(big)
    eng.set_ranges(*big.ranges)
    for i in big.img_ids:
        eng.add_image_matches(int(i), *big.flat_matches(int(i)))
    l0 = eng.stats()["n_kernel_launches"]
    reused = _outputs(eng, False, monkeypatch)
    l_reused = eng.stats()["n_kernel_launches"] - l0
    fresh_eng = _engine(big, _cfg())
    f0 = fresh_eng.stats()["n_kernel_launches"]
    fresh = _outputs(fresh_eng, False, monkeypatch)
    l_fresh = fresh_eng.stats()["n_kernel_launches"] - f0
    assert int(fresh["nodes"]["n_cand"].max()) > 32
    assert l_fresh < l_reused <= 2 * l_fresh  # one repeated pass
    _assert_same(reused, fresh)
    # the repeated pass left the exact capacity: the next run does not repeat
    l1 = eng.stats()["n_kernel_launches"]
    _assert_same(_outputs(eng, False, monkeypatch), fresh)
    assert eng.stats()["n_kernel_launches"] - l1 == l_fresh
