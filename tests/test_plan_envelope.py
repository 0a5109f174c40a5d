"""Launch plans and the size envelope, on host-only handles (device = -1: the layout and the plan are made as on a
B200 with 148 SMs, nothing is launched).

(1) Every row (problem, configuration) that test_gpu_launch_shapes.py runs must reach the code path it is there for: the
plan a handle reports ("build_plan", Model::get_index) is compared with its baseline's, with the same environment,
arguments and problem, so a change of the planner that stops a row from reaching its path fails here instead of leaving
the GPU matrix testing nothing new.  (2) The size envelope: which block
shapes are accepted and which fail at creation with code 4 and which message; keep_H = True and keep_H = False (what
spamtree() and the benchmark use) must agree on every shape.  (3) Trees from clustered data that make_tree() builds
today but the model rejects, pinned as strict xfails."""
import numpy as np
import pytest

import common
import launch_configs as lc
import shape_trees as st
import spamtree_b200 as sb

GRAM_FUSED_TAB, GRAM_CHILD_TAB = 64, 256  # st_kernels.cuh: kGramFusedTab, kGramChildTab


def _plan(pb, keep_H=False, **kw):
    g = common.product_model(pb, device=-1, keep_H=keep_H, **kw)
    try:
        return st.build_plan(g)
    finally:
        g.close()


@pytest.mark.parametrize("name,config", lc.ROWS + [(lc.CHAIN_PROBLEM, c) for c in lc.CHAIN_CONFIGS],
                         ids=[f"{p}-{c}" for p, c in lc.ROWS] + [f"chain-{c}" for c in lc.CHAIN_CONFIGS])
def test_gpu_row_reaches_its_path(name, config):
    """every row of test_gpu_launch_shapes.py runs a plan that differs from its baseline's in the way its configuration is
    there for (launch_configs.py: reach); rows of configurations that are not plan choices only need to be created"""
    c = lc.CONFIGS[config]
    p = lc.plan(name, config)
    if c["reach"] is not None:
        b = lc.plan(name, c["base"], keep_H=c["keep_H"])
        assert c["reach"](b, p), (name, config, b, p)


# paths the default plan takes on the hand-built trees (rows "shape_*-default" of the GPU matrix)
DEFAULT_PATHS = {
    "single_ring": ("p_hundreds", lambda la, lv: {x["ns"] for x in la} == {1, 2}),
    "paired_warps": ("ref_m_edges", lambda la, lv: max(x["max_npair"] for x in la) > 0),
    "gram_untabulated": ("fanout", lambda la, lv: max(v["max_children"] for v in lv) > GRAM_FUSED_TAB and
                         max(v["max_child_tiles"] for v in lv) > GRAM_CHILD_TAB),
    "gram_row_chunks": ("leaf_m_edges", lambda la, lv: any(v["max_rows"] > v["gram_rch"] for v in lv)),
    "gram_item_rounds": ("ref_m_edges", lambda la, lv: any(v["max_items"] > v["gram_threads"] and v["gram_stage_off"] > 0 for v in lv)),
    "deferred": ("fanout", lambda la, lv: lv[-1]["deferrable"] == 1),
    "wide_cta": ("leaf_m_edges", lambda la, lv: {x["threads"] for x in la} >= {256, 512}),
}


@pytest.mark.parametrize("path", sorted(DEFAULT_PATHS))
def test_default_plan_of_shape_tree_reaches_path(path):
    shape, pred = DEFAULT_PATHS[path]
    la, lv = lc.plan(f"shape_{shape}", "default", keep_H=False)
    assert pred(la, lv), (path, la, lv)


@pytest.mark.parametrize("name", sorted(st.SHAPES))
def test_shape_trees_are_accepted_and_match_the_dense_twin(name):
    """every shape of the GPU matrix is inside the envelope, and the oracle the GPU is checked against agrees with dense
    numpy on it (the generator builds what the product and the oracle read the same way)"""
    from dense_twin import Twin
    pb = st.shape_problem(name)
    for kh in (True, False):
        _plan(pb, keep_H=kh)
    if pb["limited"]:
        return
    om = common.oracle_model(pb)
    w = np.random.default_rng(1).standard_normal(pb["n"]) * .5
    om.w = w
    ok, ll, _ = om.get_loglik_comps_w(0)
    om.close()
    assert ok and abs(ll - Twin(pb).loglik(w)) <= 1e-10 * abs(ll)


OK = None
BUILD = "a block is too large for one BUILD work group"
GIBBS = "a block is too large for the Gibbs kernel's shared memory"
GRAM = "message Gram tiles do not fit the Gram kernel's shared memory"
LLW_P = "a parent set larger than 1024 rows is not supported"
CHAIN = "ancestor chains longer than 32 are not supported"
# (name, levels, expected): None = accepted, else the code-4 message
ENVELOPE = (
    [(f"leaf_m{m}", [[25], [[m]]], OK) for m in (31, 32, 33, 104, 105, 120, 121, 127, 128)] +
    [("leaf_m129", [[25], [[129]]], BUILD)] +
    [(f"ref_m{m}", [[25], [[m]], [[5]]], OK) for m in (31, 32, 33, 104, 105, st.MAX_REF_M)] +
    [(f"ref_m{m}", [[25], [[m]], [[5]]], GIBBS) for m in (st.MAX_REF_M + 1, 127, 128)] +
    [("ref_m129", [[25], [[129]], [[5]]], BUILD), ("root_m128", [[128], [[5]]], GIBBS)] +
    # parent sets: a reference block of 25 rows takes 425 parent rows, not 450; at 1024+ rows the LLW kernel's limit comes first
    [("ref_P425", st.chain(18, 25, 5), OK), ("ref_P450", st.chain(19, 25, 5), BUILD),
     ("P1024", st.chain(16, 64, 5), BUILD), ("P1040", st.chain(16, 65, 5), LLW_P)] +
    [("chain32", st.chain(32, 5, 5), OK), ("chain33", st.chain(33, 5, 5), CHAIN)] +
    # message Gram tiles of a reference block with children: m^2 summed over the block and its ancestors, 20480 doubles
    [("gram_2x101", st.chain(2, 101, 5), OK), ("gram_2x102", st.chain(2, 102, 5), GRAM),
     ("gram_3x82", st.chain(3, 82, 5), OK), ("gram_3x83", st.chain(3, 83, 5), GRAM)]
)


@pytest.mark.parametrize("name,levels,expected", ENVELOPE, ids=[e[0] for e in ENVELOPE])
def test_size_envelope(name, levels, expected):
    """accepted, or code 4 with its message at creation (before anything is launched); the same with and without keep_H.
    (leaf_m128: the deferred scheme's extra panel column would make the block one column too wide for a work group;
    the level then runs the eager scheme)"""
    pb = st.make_shape_problem(levels)
    for kh in (True, False):
        if expected is None:
            _plan(pb, keep_H=kh)
        else:
            with pytest.raises(sb.SpamTreeError) as e:
                _plan(pb, keep_H=kh)
            assert e.value.code == 4 and expected in str(e.value), (kh, str(e.value))


def test_reduced_panel_budget_rejects_at_creation():
    """a panel budget below what a block needs is an error at creation, not a launch failure (the limited q = 2 tree of
    cell 36 factorises K_uu as well and does not fit 48 KiB; it does fit 96 KiB)"""
    pb = common.make_problem(2, 2500, cell_size=36, limited=True)
    with pytest.raises(sb.SpamTreeError) as e:
        _plan(pb, smem_panel_bytes=48 * 1024)
    assert e.value.code == 4 and BUILD in str(e.value)
    la, _ = _plan(pb, smem_panel_bytes=96 * 1024)
    assert all(x["smem"] <= 96 * 1024 for x in la)


def test_deferral_falls_back_to_eager_for_a_full_width_leaf():
    """a childless level is deferred unless one of its blocks does not fit a work group with the extra column"""
    _, lv = _plan(st.make_shape_problem([[25], [[127, 7]]]))
    assert lv[-1]["deferrable"] == 1
    _, lv = _plan(st.make_shape_problem([[25], [[128, 7]]]))
    assert lv[-1]["deferrable"] == 0


def _clustered(n_clusters, per, spread, seed=0):
    rng = np.random.default_rng(seed)
    c = rng.random((n_clusters, 2))
    coords = np.repeat(c, per, axis=0) + spread * rng.standard_normal((n_clusters * per, 2))
    return coords


def _repeated_sites(n_sites, reps, seed=0):
    rng = np.random.default_rng(seed)
    return np.repeat(rng.random((n_sites, 2)), reps, axis=0)


@pytest.mark.xfail(strict=True, raises=sb.SpamTreeError,
                   reason="leaves wider than one BUILD work group (and parent sets above 1024 rows) are not supported: "
                          "clustered or repeated locations give make_tree() cells that cannot be split")
@pytest.mark.parametrize("data", ["clusters_20x1000", "sites_400x50"])
def test_clustered_data_is_accepted(data):
    coords = _clustered(20, 1000, 1e-3) if data.startswith("clusters") else _repeated_sites(400, 50)
    coords = coords[np.lexsort((coords[:, 1], coords[:, 0]))]
    n = coords.shape[0]
    y = np.random.default_rng(1).standard_normal(n)
    mv = np.ones(n, np.int64)
    t = sb.make_tree(coords, y, mv)
    csr = (t["indexing_ptr"], t["indexing_idx"], t["parents_ptr"], t["parents_idx"], t["children_ptr"], t["children_idx"])
    pb = {"d": {"y": y, "X": np.ones((n, 1)), "coords": coords, "mv_id": mv}, "tree": t, "csr": csr,
          "theta": np.array([2.3, 1.0, 1.0, 6.0]), "beta": np.zeros(1), "tausq": 0.1}
    try:
        _plan(pb, keep_H=False)
    except sb.SpamTreeError as e:
        assert e.code == 4, str(e)
        raise
