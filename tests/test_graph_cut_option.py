"""CPU checks of the graph-cut choice: PHMRF_GRAPH_CUT reaches the model as graph_cut, a bad value is refused,
and the model refuses an unknown graph_cut."""
import numpy as np
import pytest

from phylo_hmrf_b200 import cli


def _run_with_stub(tmp_path, monkeypatch):
    from phylo_hmrf_b200 import hmrf
    (tmp_path / "edge.1.txt").write_text("0\t1\n1\t2\n1\t3\n")
    stem = "50Kb.observed.0"
    np.save(tmp_path / ("data.%s.npy" % stem), np.ones((6, 2)))
    ev = np.empty(1, dtype=object)
    ev[0] = np.zeros((4, 3))
    np.save(tmp_path / ("edgelist.%s.npy" % stem), ev, allow_pickle=True)
    np.savetxt(tmp_path / ("lenvec.%s.txt" % stem), np.asarray([[6, 0, 6, 3, 3, 0, 0, 0, 1, 21]]), fmt='%d',
               delimiter='\t')
    seen = {}

    class Stub:
        def __init__(self, **kw):
            seen["model"] = kw

        def fit_accumulate_test(self, samples, len_vec, threshold, filename, miter):
            return (np.zeros(1),) * 4 + (np.zeros(1), np.zeros(1), np.zeros(6))

        def close(self):
            pass

    monkeypatch.setattr(hmrf, "phyloHMRF", Stub)
    monkeypatch.chdir(tmp_path)
    cli.run(cli.parse_args(["-p", str(tmp_path), "--output", str(tmp_path), "--reload", "1"]))
    return seen["model"]


@pytest.mark.parametrize("value,expect", [(None, "host"), ("host", "host"), ("device", "device")])
def test_environment_selects_the_graph_cut(tmp_path, monkeypatch, value, expect):
    if value is None:
        monkeypatch.delenv("PHMRF_GRAPH_CUT", raising=False)
    else:
        monkeypatch.setenv("PHMRF_GRAPH_CUT", value)
    assert _run_with_stub(tmp_path, monkeypatch)["graph_cut"] == expect


def test_bad_environment_value_is_refused(tmp_path, monkeypatch):
    monkeypatch.setenv("PHMRF_GRAPH_CUT", "gpu")
    with pytest.raises(SystemExit, match="PHMRF_GRAPH_CUT"):
        _run_with_stub(tmp_path, monkeypatch)


def test_model_refuses_an_unknown_graph_cut():
    from phylo_hmrf_b200.hmrf import phyloHMRF
    with pytest.raises(ValueError, match="graph_cut"):
        phyloHMRF(10, 2, graph_cut="gpu")


def test_swap_supported():
    from phylo_hmrf_b200.engine import swap_supported
    potts = (3 * (1 - np.eye(4))).astype(np.int32)
    assert swap_supported(potts, 0.0)
    assert not swap_supported(potts, -1e-3)
    assert not swap_supported(np.asarray([[0, 1], [1, 5]], np.int32), 1.0)
    assert swap_supported(np.asarray([[0, 3], [0, 0]], np.int32), 1.0)    # asymmetric, still submodular
