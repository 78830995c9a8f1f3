"""Host-side data loading (phylo_hmrf_b200/loader.py) against fixtures produced by the reference's own
functions on a mini data set (tests/golden/make_golden_prep.py::make_loader_cases), plus the
per-chromosome assembly with the GPU-backed stages replaced by oracle stand-ins."""
import os
import sys

import numpy as np
import pytest

from oracle import prep_oracle as po

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "golden"))
from make_golden_prep import write_loader_inputs  # noqa: E402

G = np.load(os.path.join(HERE, "golden", "loader_cases.npz"))
SPECIES = ["sp0", "sp1", "sp2"]


def test_multi_species_alignment_matches_the_reference(tmp_path):
    from phylo_hmrf_b200 import loader
    dirs = write_loader_inputs(str(tmp_path), G)
    res = int(G["resolution"])
    data = loader.multi_contact_matrix3A("3", res, str(tmp_path / "chrom.sizes"), dirs, SPECIES, "", 0)
    assert list(data) == [0, 1, 2] + SPECIES
    np.testing.assert_array_equal(np.asarray(data.loc[:, [0, 1, 2]]), G["aligned_position"])
    np.testing.assert_array_equal(np.asarray(data.loc[:, SPECIES], dtype=np.float64), G["aligned_x"])
    assert (G["aligned_x"] == -1).any(), "fixture must exercise the NaN -> -1 rule"
    assert loader.multi_contact_matrix3A("9", res, str(tmp_path / "chrom.sizes"), dirs, SPECIES, "", 0) == -1
    assert loader.multi_contact_matrix3A("1", res, str(tmp_path / "chrom.sizes"), dirs, SPECIES, "", 0) is False


def test_subregion1_matches_the_reference(tmp_path):
    from phylo_hmrf_b200 import loader
    write_loader_inputs(str(tmp_path), G)
    f = str(tmp_path / "chr3.synteny.txt")
    region_list, list1 = loader.subregion1(f, 3, int(G["resolution"]), [np.array([90279522, 93797661])], 0)
    np.testing.assert_array_equal(np.asarray([list(map(int, r)) for r in region_list]), G["region_list"])
    np.testing.assert_array_equal(np.asarray([list(map(int, r)) for r in list1]), G["list1"])
    _, list1 = loader.subregion1(f, 3, int(G["resolution"]), [], 0)
    np.testing.assert_array_equal(np.asarray([list(map(int, r)) for r in list1]), G["list1_nosplit"])
    # a single-line file (numpy returns a 1-D array): one diagonal region
    g = str(tmp_path / "one.txt")
    np.savetxt(g, np.array([[5, 50, 45]]), fmt="%d", delimiter="\t")
    _, one = loader.subregion1(g, 7, 10, [], 0)
    assert [list(map(int, r)) for r in one] == [[5, 50, 5, 50, 45, 45, 0, 0, 7]]


def test_chromosome_assembly(tmp_path, monkeypatch):
    """load_data_chromosome2 (utility.py:267-468): regions in id order, cumulative sample offsets inserted
    at len_vec[1:3], chromosome offsets added on top; GPU stages replaced by oracle stand-ins."""
    from phylo_hmrf_b200 import loader, utility

    def fake_norm(x1, x_min, x_max, device=0):
        y, vec1, lo, hi = po.normalize_feature(x1, x_min, x_max)
        return po.log_transform(y), vec1, lo, hi

    def fake_unsym(value, pos, f1, f2, nn, sigma, type_id, fm, fp1, fp2, device=0, want_image=True):
        data1, _, pos_idx, _ = po.image_pipeline_diag(value, pos[:, :2], filter_mode=-1)
        return data1, None, pos_idx, np.full((3, 3), 1.0)

    def fake_sym(value, pos, f1, f2, nn, sigma, type_id, fm, fp1, fp2, device=0, want_image=True):
        p = pos[:, :2]
        n1, n2 = p[:, 0].max() - p[:, 0].min() + 1, p[:, 1].max() - p[:, 1].min() + 1
        return np.zeros((n1 * n2, value.shape[1])), None, None, np.full((2, 3), 2.0)

    monkeypatch.setattr(utility, "normalize_log_feature", fake_norm)
    monkeypatch.setattr(utility, "write_matrix_image_Ctrl_unsym1", fake_unsym)
    monkeypatch.setattr(utility, "write_matrix_image_Ctrl_sym1", fake_sym)
    dirs = write_loader_inputs(str(tmp_path), G)
    res = int(G["resolution"])
    samples, len_vec, edges = loader.load_data_chromosome2([3], -1, -1, res, 8, 0, 0.0, 0, str(tmp_path / "chrom.sizes"),
                                                           dirs, SPECIES, str(tmp_path))
    assert len(len_vec) == len(edges) == len(G["list1"]) == 4      # 3 pairs of the split block + 1 block
    off = 0
    for lv, row in zip(len_vec, G["list1"]):
        n = lv[0]
        assert lv[1] == off and lv[2] == off + n and lv[7] == row[6] and lv[9] == 3  # [6]: synteny block id
        assert lv[8] == (1 if (row[0] == row[2] and row[1] == row[3]) else 0)
        off += n
    assert samples.shape == (off, 3)
    # diagonal regions only
    s2, lv2, e2 = loader.load_data_chromosome2([3], -1, -1, res, 8, 0, 0.0, 1, str(tmp_path / "chrom.sizes"), dirs,
                                               SPECIES, str(tmp_path))
    assert [lv[8] for lv in lv2] == [1, 1, 1] and s2.shape[0] == lv2[-1][2]


def test_quantiles_match_the_reference(tmp_path):
    from phylo_hmrf_b200 import loader
    dirs = write_loader_inputs(str(tmp_path), G)
    q = loader.quantile_contact_vec(["3"], int(G["resolution"]), str(tmp_path / "chrom.sizes"), dirs, SPECIES)
    np.testing.assert_array_equal(q, G["quantiles"])
