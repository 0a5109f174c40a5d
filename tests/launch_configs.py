"""The launch-plan configurations test_gpu_launch_shapes.py runs, the problems it runs each one on, and what each one must
change in the plan relative to its baseline configuration on every one of those problems.  test_plan_envelope.py checks
the latter on host-only handles ("build_plan", Model::get_index): a row whose configuration stops reaching its path fails
on the CPU instead of running the baseline's plan on the GPU once more."""
import os

import common
import shape_trees as st

PROBLEMS = {
    "q1_n625": lambda: common.make_problem(1, 625),
    "q3_n3000_imbalanced": lambda: common.make_problem(3, 3000, proportions=(.6, .3, .1)),
    "q2_n2500_cell36_limited": lambda: common.make_problem(2, 2500, cell_size=36, limited=True),
    "q5_n4000": lambda: common.make_problem(5, 4000, missing=.15),
}
PROBLEMS.update({f"shape_{k}": (lambda k=k: st.shape_problem(k)) for k in st.SHAPES})
MAKE_TREE = [p for p in PROBLEMS if not p.startswith("shape_")]

_pb = {}


def problem(name):
    if name not in _pb:
        _pb[name] = PROBLEMS[name]()
    return _pb[name]


def _nn(p):
    return max(x["max_nn"] for x in p[0])


def _count(p, f):
    return sum(1 for x in p[0] if f(x))


def _lcount(p, f):
    return sum(1 for v in p[1] if f(v))


# name -> env: environment read at handle creation; kw: constructor arguments; bitwise: must reproduce the baseline bit for
# bit; base: the configuration it is compared with; keep_H: the handle whose plan shows the change; reach(base plan,
# plan): the change, on every problem of its rows (None: not a plan choice, see the comment)
CONFIGS = {
    "default": dict(env={}, kw={}, bitwise=True, base=None, keep_H=True, reach=None),
    # groups of many siblings (wider CTAs, paired warps)
    "spread0": dict(env={"ST_SPREAD": "0"}, kw={}, bitwise=False, base="default", keep_H=True,
                    reach=lambda b, p: _nn(p) > _nn(b)),
    # multi-block groups of more than 104 columns
    "spread0_maxcols128": dict(env={"ST_SPREAD": "0", "ST_MAX_COLS": "128"}, kw={}, bitwise=False, base="spread0", keep_H=True,
                               reach=lambda b, p: _count(p, lambda x: x["max_nn"] > 1 and x["max_ncp"] > 104) >
                               _count(b, lambda x: x["max_nn"] > 1 and x["max_ncp"] > 104)),
    # one block per group where the spread rule alone puts several (without ST_SPREAD=0 the groups of a level with fewer
    # blocks than SMs hold one block already)
    "spread0_maxcols8": dict(env={"ST_SPREAD": "0", "ST_MAX_COLS": "8"}, kw={}, bitwise=False, base="spread0", keep_H=True,
                             reach=lambda b, p: _count(b, lambda x: x["max_nn"] > 1 and x["max_ncp"] > 8) > 0 and
                             _count(p, lambda x: x["max_nn"] > 1 and x["max_ncp"] > 8) == 0),
    # ring depth: the single ring where the default has a double one, and the reverse
    "ns1": dict(env={"ST_BUILD_NS": "1"}, kw={}, bitwise=True, base="default", keep_H=True,
                reach=lambda b, p: _count(b, lambda x: x["ns"] == 2) > 0 and _count(p, lambda x: x["ns"] == 2) == 0),
    "ns2": dict(env={"ST_BUILD_NS": "2"}, kw={}, bitwise=True, base="default", keep_H=True,
                reach=lambda b, p: _count(b, lambda x: x["ns"] == 1) > 0 and _count(p, lambda x: x["ns"] == 1) == 0),
    # reduced panel budgets: every launch within the budget where the baseline has launches above it
    "smem48k": dict(env={}, kw={"smem_panel_bytes": 48 * 1024}, bitwise=False, base="default", keep_H=True,
                    reach=lambda b, p: _count(b, lambda x: x["smem"] > 48 * 1024) > 0 and _count(p, lambda x: x["smem"] > 48 * 1024) == 0),
    "spread0_smem96k": dict(env={"ST_SPREAD": "0"}, kw={"smem_panel_bytes": 96 * 1024}, bitwise=False, base="spread0", keep_H=True,
                            reach=lambda b, p: _count(b, lambda x: x["smem"] > 96 * 1024) > 0 and _count(p, lambda x: x["smem"] > 96 * 1024) == 0),
    # Gram rows staged in more chunks than by default
    "gram_room1": dict(env={"ST_GRAM_ROOM": "1"}, kw={}, bitwise=True, base="default", keep_H=True,
                       reach=lambda b, p: _lcount(p, lambda v: v["max_rows"] > v["gram_rch"]) > _lcount(b, lambda v: v["max_rows"] > v["gram_rch"])),
    # (not a plan choice: every level launch but a stream's first is a programmatic dependent launch unless ST_PDL=0)
    "pdl0": dict(env={"ST_PDL": "0"}, kw={}, bitwise=True, base="default", keep_H=True, reach=None),
    # the eager scheme at the childless level of a keep_H = False handle
    "defer0": dict(env={"ST_DEFER": "0"}, kw={}, bitwise=True, base="default", keep_H=False,
                   reach=lambda b, p: _lcount(b, lambda v: v["deferrable"]) > 0 and _lcount(p, lambda v: v["deferrable"]) == 0),
    # device-resident chain only (the host-driven operations run every launch on one stream)
    "overlap0": dict(env={"ST_OVERLAP": "0"}, kw={}, bitwise=True, base="default", keep_H=False,
                     reach=lambda b, p: _lcount(b, lambda v: v["early"]) > 0 and _lcount(p, lambda v: v["early"]) == 0),
    # (device-resident chain only, and not a plan choice: LLW runs on the second stream in every iteration that samples w and theta)
    "llw_overlap1": dict(env={"ST_LLW_OVERLAP": "1"}, kw={}, bitwise=True, base="default", keep_H=False, reach=None),
}

# host-driven rows: (problem, configuration)
ROWS = (
    [(p, "default") for p in PROBLEMS] +
    [(p, "spread0") for p in MAKE_TREE + ["shape_leaf_m_edges", "shape_fanout", "shape_fanout_q3", "shape_nan_siblings",
                                          "shape_limited_fanout", "shape_p_edges", "shape_ref_m_edges"]] +
    [(p, "spread0_maxcols128") for p in ["q2_n2500_cell36_limited", "shape_fanout"]] +
    [(p, "spread0_maxcols8") for p in ["q1_n625", "shape_fanout", "shape_nan_siblings"]] +
    [(p, "ns1") for p in MAKE_TREE + ["shape_ref_m_edges"]] +
    [(p, "ns2") for p in ["shape_p_hundreds"]] +
    [(p, "smem48k") for p in ["q3_n3000_imbalanced", "q5_n4000", "shape_chain32"]] +
    [(p, "spread0_smem96k") for p in ["q5_n4000", "shape_fanout"]] +
    [(p, "gram_room1") for p in ["q3_n3000_imbalanced", "q5_n4000", "shape_fanout", "shape_ref_m_edges"]] +
    [(p, "pdl0") for p in MAKE_TREE] +
    [(p, "defer0") for p in ["q3_n3000_imbalanced", "q5_n4000", "shape_fanout"]]
)
# the device-resident chain: q = 3, n = 3000, against the default chain (bitwise) or against the host replay under the
# same configuration (spread0, whose reduction order differs from the default's)
CHAIN_PROBLEM = "q3_n3000_imbalanced"
CHAIN_CONFIGS = ["pdl0", "overlap0", "llw_overlap1", "defer0", "spread0"]


def plan(name, config, keep_H=None, which="build_plan"):
    """the plan of a host-only handle of problem `name` under `config` (environment set for the creation only):
    shape_trees.build_plan, or with which="build_groups" the (level, first slot, nn, NCp, threads, npair) of every work group"""
    c = CONFIGS[config]
    old = {k: os.environ.get(k) for k in c["env"]}
    os.environ.update(c["env"])
    try:
        g = common.product_model(problem(name), device=-1, keep_H=c["keep_H"] if keep_H is None else keep_H, **c["kw"])
    finally:
        for k, v in old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v
    try:
        return st.build_plan(g) if which == "build_plan" else g.index(which).reshape(-1, 6)
    finally:
        g.close()
