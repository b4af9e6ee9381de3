"""Runner-level drop-in (BASELINE.json configs[0]: the reference plumbing on a 10-image scene; SURVEY.md §8d config 1:
V=10, L=800, N=9, K=10 through limap.runners.line_triangulation with load_det / load_match artefacts).

  * CPU: the REFERENCE'S OWN runner file, src/limap/runners/line_triangulation.py, loaded by path and executed
    UNMODIFIED against this repository's `limap` package (base, triangulation, merging, optimize, vplib, util.io,
    runners, visualize), with the three engine classes replaced by oracle-backed stand-ins. What it returned and wrote is
    stored in tests/golden/ref/runner_line_triangulation.npz (recorded by tests/golden/make_ref_golden.py with
    LIMAP_REFERENCE pointing at a LIMAP source tree). This repository's own runner mirror (limap_b200/runners.py) on the
    same artefacts must reproduce it: same tracks, same refined lines, same files on disk, same [Track Report].
  * GPU: the runner mirror with the real CUDA engines against the same mirror on the oracle stand-ins: track
    membership bit-exact, refined endpoints 1e-4, [Track Report] equal.
Together: reference runner == mirror (same surface), mirror on CUDA == mirror on the oracle (same arithmetic)."""
import importlib.util
import os
import sys
import types

import numpy as np
import pytest

from limap_b200.config import default_runner_config
from limap_b200.synth import CONFIGS, make_scene

from runner_utils import imagecols_of, install_oracle_backend, summarize, write_artifacts
from ref_golden import reference as _reference

RUNNER_FILES = ("image_list.txt", "metainfos.txt", "alltracks.txt", "finaltracks/track_0.txt", "triangulated_lines_nv4.obj")


def _reference_tree_file(rel):
    """A file of the LIMAP source tree at $LIMAP_REFERENCE (read only when recording the golden outputs)."""
    return os.path.join(os.environ["LIMAP_REFERENCE"], rel)


def _scene(small):
    if small:
        return make_scene(V=8, L=120, N=5, K=6, seed=51)
    return make_scene(**CONFIGS["hypersim10"])


def _cfg(tmp, sc, **over):
    cfg = default_runner_config(output_dir=str(tmp / "out"), load_dir=str(tmp / "artefacts"), n_neighbors=9, **over)
    write_artifacts(sc, cfg, cfg["load_dir"])
    return cfg


def _run_mirror(cfg, sc):
    import copy
    import limap.runners as runners
    return runners.line_triangulation(copy.deepcopy(cfg), imagecols_of(sc), neighbors=dict(sc.neighbors), ranges=sc.ranges)


def _report(tracks):
    import limap.visualize as vis
    return vis.Open3DTrackVisualizer(tracks).track_report()


def _record_reference_runner(tmp_path, monkeypatch, capsys, sc, cfg):
    import copy
    # the only names the reference runner imports that are not part of the hot path: pycolmap (logging) -- stubbed
    pyc = types.ModuleType("pycolmap")
    pyc.logging = types.SimpleNamespace(info=lambda *a, **k: None, warning=lambda *a, **k: None, error=lambda *a, **k: None)
    monkeypatch.setitem(sys.modules, "pycolmap", pyc)
    monkeypatch.setitem(sys.modules, "pycolmap.logging", pyc.logging)
    import limap  # noqa: F401  (alias package: limap.X -> limap_b200.X)
    path = _reference_tree_file("src/limap/runners/line_triangulation.py")
    spec = importlib.util.spec_from_file_location("reference_line_triangulation", path)
    ref_mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(ref_mod)
    with open(path) as f:
        assert "def line_triangulation(cfg, imagecols, neighbors=None, ranges=None):" in f.read()
    cfg_ref = copy.deepcopy(cfg)
    cfg_ref["output_dir"] = str(tmp_path / "out_ref")
    ref_tracks = ref_mod.line_triangulation(cfg_ref, imagecols_of(sc), neighbors=dict(sc.neighbors), ranges=sc.ranges)
    assert "[Track Report]" in capsys.readouterr().out
    members, lines = summarize(ref_tracks)
    out = dict(track_off=np.concatenate([[0], np.cumsum([len(m) for m in members])]),
               members=np.asarray([x for m in members for x in m], np.int32).reshape(-1, 2), lines=lines,
               report=np.asarray(_report(ref_tracks)),
               imagecols_npy=np.asarray((tmp_path / "out_ref" / "imagecols.npy").exists()))
    for k, rel in enumerate(RUNNER_FILES):
        out[f"file_{k}"] = np.frombuffer((tmp_path / "out_ref" / rel).read_bytes(), np.uint8)
    return out


def test_reference_runner_file_runs_unmodified_on_this_surface(tmp_path, monkeypatch, capsys):
    install_oracle_backend(monkeypatch)
    sc = _scene(small=True)
    cfg = _cfg(tmp_path, sc)
    r = _reference("runner_line_triangulation", lambda: _record_reference_runner(tmp_path, monkeypatch, capsys, sc, cfg))
    my_tracks = _run_mirror(cfg, sc)
    m_my, l_my = summarize(my_tracks)
    off = r["track_off"]
    m_ref = [tuple(map(tuple, r["members"][off[k]:off[k + 1]].tolist())) for k in range(len(off) - 1)]
    assert len(m_ref) > 20 and m_ref == m_my
    assert np.array_equal(r["lines"], l_my)  # same backend, same call sequence: bit-identical
    assert tuple(r["report"].tolist()) == _report(my_tracks)
    # the files a user finds afterwards
    assert bool(r["imagecols_npy"]) and (tmp_path / "out" / "imagecols.npy").exists()
    for k, rel in enumerate(RUNNER_FILES):
        assert (tmp_path / "out" / rel).read_bytes() == r[f"file_{k}"].tobytes(), rel
    import limap.util.io as limapio
    back, cfg_back, ic_back, segs_back = limapio.read_folder_linetracks_with_info(str(tmp_path / "out" / "finaltracks"))
    assert len(back) == len(my_tracks) and ic_back.NumImages() == len(sc.img_ids) and len(segs_back) == len(sc.img_ids)


@pytest.mark.gpu
def test_runner_mirror_cuda_equals_oracle_backend_hypersim10(tmp_path, monkeypatch):
    sc = _scene(small=False)  # V=10, L=800, N=9, K=10: the configs[0] stand-in
    cfg = _cfg(tmp_path, sc)
    gpu_tracks = _run_mirror(cfg, sc)
    rep_gpu = _report(gpu_tracks)
    with monkeypatch.context() as mp:
        install_oracle_backend(mp)
        cfg2 = dict(cfg, output_dir=str(tmp_path / "out_cpu"))
        cpu_tracks = _run_mirror(cfg2, sc)
    (m_g, l_g), (m_c, l_c) = summarize(gpu_tracks), summarize(cpu_tracks)
    assert len(m_c) > 100 and m_g == m_c
    d = np.minimum(np.abs(l_g - l_c).max(1), np.abs(l_g - l_c[:, [3, 4, 5, 0, 1, 2]]).max(1))
    assert d.max() <= 1e-4, d.max()
    assert rep_gpu == _report(cpu_tracks) and rep_gpu[0] == len(m_c)
    assert (tmp_path / "out" / "finaltracks" / "track_0.txt").exists()


def _record_reference_linebase_test():
    """The one test of the reference's own suite that touches a hot-path type (tests/base/test_linebase.py::test_line2d),
    run unmodified against `import limap` = this repository's alias package, with Line2d recording what it is asked and
    numpy.testing recording what is compared: the known-answer vectors of that test."""
    import numpy.testing as npt
    import limap
    made, checks = [], []
    line2d = limap.base.Line2d

    def recording_line2d(start, end):
        made.append(np.concatenate([np.asarray(start, float), np.asarray(end, float)]))
        return line2d(start, end)

    def recording_allclose(actual, desired, rtol=1e-7, atol=0):
        checks.append((np.atleast_1d(np.asarray(desired, float)), rtol, atol))
        npt.assert_allclose(actual, desired, rtol=rtol, atol=atol)
    spec = importlib.util.spec_from_file_location("ref_test_linebase", _reference_tree_file("tests/base/test_linebase.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    assert mod.limap is limap and limap.base.__name__ == "limap_b200.base"
    mod.limap = types.SimpleNamespace(base=types.SimpleNamespace(Line2d=recording_line2d))
    mod.npt = types.SimpleNamespace(assert_allclose=recording_allclose)
    mod.test_line2d()
    assert len(made) == 1 and len(checks) == 2
    return dict(line=made[0], length=checks[0][0], direction=checks[1][0],
                tol=np.array([[c[1], c[2]] for c in checks]))


def test_reference_own_linebase_test_passes_on_the_mirror():
    """tests/base/test_linebase.py::test_line2d of the reference's own suite on the mirror: Line2d((0, 0), (1, 1)) has
    length sqrt(2) and direction (1, 1) / sqrt(2), with that test's tolerances (tests/golden/ref/linebase_test_line2d.npz)."""
    import numpy.testing as npt
    import limap
    assert limap.base.__name__ == "limap_b200.base"
    r = _reference("linebase_test_line2d", _record_reference_linebase_test)
    line = limap.base.Line2d(r["line"][:2], r["line"][2:])
    npt.assert_allclose(line.length(), r["length"][0], rtol=r["tol"][0, 0], atol=r["tol"][0, 1])
    npt.assert_allclose(line.direction(), r["direction"], rtol=r["tol"][1, 0], atol=r["tol"][1, 1])
