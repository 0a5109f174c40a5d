"""New rows attached to a built tree (st_tree_attach) follow the rule of the tree's own prediction level: attaching the
missing rows of a tree to that tree gives back its missing level bit for bit — the same partition into blocks and the
parent lists of make_edges / make_edges_limited.  Host-only, no GPU."""
import numpy as np
import pytest

import spamtree_b200 as sb
from spamtree_b200 import synth


def _data(q, n, proportions=None, seed=2021):
    return synth.make_data(q, n, proportions, missing=0.1, seed=seed)


def _check_missing_level(d, limited=False, **kw):
    miss = np.isnan(d["y"])
    assert miss.any()
    t = sb.make_tree(d["coords"], d["y"], d["mv_id"], coords_new=d["coords"][miss], mv_id_new=d["mv_id"][miss],
                     limited_tree=limited, **kw)
    new = t["new"]
    blocks = t["blocking"][miss]
    groups = new["group"]
    # the same partition, groups numbered like the blocks (rank of the parent block)
    g2b = {}
    for g, b in zip(groups, blocks):
        assert g2b.setdefault(int(g), int(b)) == int(b)
    assert len(g2b) == new["n_groups"] == np.unique(blocks).size
    assert sorted(g2b) == list(range(new["n_groups"]))
    assert all(g2b[g] < g2b[g + 1] for g in range(new["n_groups"] - 1))
    # the parent lists of the missing blocks
    ne = np.unique(t["blocking"][np.isfinite(d["y"])])
    e = (sb.make_edges_limited if limited else sb.make_edges)(t["parchi_map"], ne, t["res_is_ref"])
    for g in range(new["n_groups"]):
        got = new["parents_idx"][new["parents_ptr"][g]:new["parents_ptr"][g + 1]]
        assert np.array_equal(got, e["parents"][g2b[g] - 1]), g
        assert got.size >= 1
    return t


@pytest.mark.parametrize("case", ["q1_n625", "q3_n3000_imbalanced", "no_same_margin", "finite_depth", "limited",
                                  "limited_q3"])
def test_attaching_the_missing_rows_gives_the_missing_level(case):
    if case == "q1_n625":
        _check_missing_level(_data(1, 625))
    elif case == "q3_n3000_imbalanced":
        _check_missing_level(_data(3, 3000, (.6, .3, .1)))
    elif case == "no_same_margin":
        _check_missing_level(_data(3, 3000, (.6, .3, .1)), cherrypick_same_margin=False)
    elif case == "finite_depth":
        d = _data(2, 2000)
        t = _check_missing_level(d, tree_depth=2)
        assert list(t["res_is_ref"][-2:]) == [0, 0]  # a leftover level, then the missing level
        assert np.unique(t["res"]).size >= 4
    elif case == "limited":
        _check_missing_level(_data(1, 625), limited=True)
    else:
        _check_missing_level(_data(3, 1500), limited=True, tree_depth=3)


def test_margin_without_targets_falls_back_to_any_margin():
    d = _data(1, 625)
    rng = np.random.default_rng(3)
    cn = rng.random((200, 2))
    a = sb.make_tree(d["coords"], d["y"], d["mv_id"], coords_new=cn, mv_id_new=np.ones(200, np.int64))["new"]
    b = sb.make_tree(d["coords"], d["y"], d["mv_id"], coords_new=cn, mv_id_new=np.full(200, 7, np.int64))["new"]
    for k in ("group", "parents_ptr", "parents_idx"):
        assert np.array_equal(a[k], b[k])


def test_make_tree_without_new_rows_is_unchanged():
    d = _data(3, 1500)
    rng = np.random.default_rng(4)
    a = sb.make_tree(d["coords"], d["y"], d["mv_id"])
    b = sb.make_tree(d["coords"], d["y"], d["mv_id"], coords_new=rng.random((50, 2)) * 3 - 1,
                     mv_id_new=rng.integers(1, 4, 50))
    assert "new" not in a and set(b) == set(a) | {"new"}
    for k in a:
        assert np.array_equal(np.asarray(a[k]), np.asarray(b[k]), equal_nan=True), k
    assert b["new"]["group"].shape == (50,)


def test_no_new_rows_and_bad_input():
    d = _data(1, 625)
    t = sb.make_tree(d["coords"], d["y"], d["mv_id"], coords_new=np.zeros((0, 2)))["new"]
    assert t["n_groups"] == 0 and t["group"].size == 0 and list(t["parents_ptr"]) == [0]
    with pytest.raises(sb.SpamTreeError):
        sb.make_tree(d["coords"], d["y"], d["mv_id"], coords_new=np.array([[0.5, np.nan]]))
    with pytest.raises(sb.SpamTreeError):
        sb.make_tree(d["coords"], d["y"], d["mv_id"], coords_new=np.zeros((3, 2)), mv_id_new=np.ones(2, np.int64))
