"""Hand-built trees of chosen block shapes, for the tests that drive the kernels' launch plans to their edges.

make_tree() gives blocks of about cell_size rows with about four children each, so the plan the kernels run under (work
group sizes, CTA widths, tabulated or untabulated Gram lookups, register or general factorisations) is whatever such trees
happen to need.  make_shape_problem() builds the tree block by block instead and returns the problem dict of
common.make_problem, so product_model, oracle_model, dense_twin.Twin and block_truth_ld all take it."""
import numpy as np

from spamtree_b200 import synth


def make_shape_problem(levels, q=1, limited=False, seed=0, tausq=0.1):
    """levels[0]: row counts of the root blocks; levels[i] (i >= 1): for each block of level i-1 in order, the list of the
    row counts of its children.  A negative count is a block of that many rows whose y are all NaN: a prediction block,
    which must be childless.  Levels 0 .. L-2 are reference levels and level L-1 the non-reference one; every level must
    hold an observed block.  The parent set of a block is its ancestor chain, root first (limited: the direct parent only),
    and a block's children list holds its observed descendants (make_edges / make_edges_limited).

    Every block's rows are spread over the unit square: the locations are the cells of a jittered grid (at least half a
    cell apart), shuffled and handed out block by block, so a parent set of any size stays well conditioned.  q = 3 puts
    the outcomes of a block on shared locations, three rows per location."""
    rng = np.random.default_rng(seed)
    sizes, parent, level = [], [], []
    prev = []
    for lev, spec in enumerate(levels):
        cur = []
        if lev == 0:
            spec = [list(spec)]
        elif len(spec) != len(prev):
            raise ValueError(f"level {lev}: {len(spec)} child lists for {len(prev)} blocks of level {lev - 1}")
        for i, kids in enumerate(spec):
            pa = -1 if lev == 0 else prev[i]
            if kids and pa >= 0 and sizes[pa] < 0:
                raise ValueError("an all-NaN block cannot have children")
            for m in kids:
                if m == 0:
                    raise ValueError("empty block")
                cur.append(len(sizes))
                sizes.append(int(m))
                parent.append(pa)
                level.append(lev)
        prev = cur
    nb, L = len(sizes), len(levels)
    level = np.asarray(level)
    obs_blk = np.asarray(sizes) > 0
    if any(not obs_blk[level == lv].any() for lv in range(L)):
        raise ValueError("every level needs an observed block")
    m_abs = np.abs(sizes)
    chain = []
    for u in range(nb):
        c, a = [], parent[u]
        while a >= 0:
            c.append(a)
            a = parent[a]
        chain.append(c[::-1])
    pars = [c[-1:] if limited else c for c in chain]
    kids = [[] for _ in range(nb)]
    for u in range(nb):
        if obs_blk[u]:
            for a in pars[u]:
                kids[a].append(u)
    # rows: block by block; locations from a shuffled jittered grid
    nloc_blk = [-(-int(m) // q) for m in m_abs]
    nloc = int(sum(nloc_blk))
    g = int(np.ceil(np.sqrt(nloc)))
    cells = rng.permutation(g * g)[:nloc]
    loc = (np.stack([cells % g, cells // g], axis=1) + 0.25 + 0.5 * rng.random((nloc, 2))) / g
    n = int(m_abs.sum())
    coords, mv_id, rows_of = np.zeros((n, 2)), np.zeros(n, np.int64), []
    r0 = l0 = 0
    for u in range(nb):
        m = int(m_abs[u])
        i = np.arange(m)
        coords[r0:r0 + m] = loc[l0 + i // q]
        mv_id[r0:r0 + m] = 1 + i % q
        rows_of.append(np.arange(r0, r0 + m, dtype=np.int64))
        r0, l0 = r0 + m, l0 + nloc_blk[u]
    if q > 1 and np.unique(mv_id[np.repeat(obs_blk, m_abs)]).size < q:
        raise ValueError("some outcome has no observed row")
    X = rng.standard_normal((n, 3))
    y = X @ np.array([-1.0, .5, 1.0]) + np.sin(4 * coords[:, 0]) * np.cos(3 * coords[:, 1]) + 0.3 * mv_id + np.sqrt(.1) * rng.standard_normal(n)
    y[~np.repeat(obs_blk, m_abs)] = np.nan

    def csr(lists):
        ptr = np.zeros(len(lists) + 1, np.int64)
        ptr[1:] = np.cumsum([len(a) for a in lists])
        idx = np.concatenate([np.asarray(a, np.int64) for a in lists]) if ptr[-1] else np.zeros(0, np.int64)
        return ptr, idx

    ip, ii = csr(rows_of)
    pp, pi = csr(pars)
    cp, ci = csr([sorted(k) for k in kids])
    tree = {"indexing_ptr": ip, "indexing_idx": ii, "parents_ptr": pp, "parents_idx": pi, "children_ptr": cp, "children_idx": ci,
            "block_names": np.arange(1, nb + 1, dtype=np.float64), "block_groups": (level + 1).astype(np.float64),
            "res_is_ref": np.array([1] * (L - 1) + [0], np.int64), "n_blocks": nb}
    d = {"y": y, "X": X, "coords": coords, "mv_id": mv_id, "q": q, "n": n}
    return {"d": d, "tree": tree, "csr": (ip, ii, pp, pi, cp, ci), "theta": synth.theta_for(q), "beta": np.zeros(3),
            "tausq": tausq, "q": q, "n": n, "limited": bool(limited)}


def chain(depth, m, leaf):
    """one reference block per level, `depth` reference levels of m rows, then a single leaf: parent sets grow to
    depth * m rows and the chain to `depth` ancestors"""
    return [[m]] + [[[m]]] * (depth - 1) + [[[leaf]]]


def build_plan(model):
    """the "build_plan" record of a handle (Model::get_index): (launches, levels) as lists of dicts"""
    r = model.index("build_plan")
    nl, nv = int(r[0]), int(r[1])
    lk = ("level", "mode", "groups", "ns", "threads", "smem", "max_nn", "max_ncp", "max_npair")
    vk = ("deferrable", "early", "gram_rch", "max_rows", "gram_stage_off", "gram_threads", "max_children", "max_child_tiles", "max_items")
    la = r[2:2 + 9 * nl].reshape(nl, 9)
    lv = r[2 + 9 * nl:2 + 9 * nl + 9 * nv].reshape(nv, 9)
    assert r.size == 2 + 9 * (nl + nv)
    return [dict(zip(lk, map(int, x))) for x in la], [dict(zip(vk, map(int, x))) for x in lv]


def _mixed_fanout():
    """two parents at depth 3 (three ancestors: four Gram tiles each) with 66 and 17 children; every other child is a
    reference block with a leaf of its own (non-fused), the rest are childless (fused into the parent)"""
    return [[25], [[20]], [[15]], [[12, 12]], [[6] * 66, [6] * 17], [[4] if i % 2 == 0 else [] for i in range(66 + 17)]]


EDGE_M = [1, 2, 5, 8, 9, 16, 17, 31, 32, 33, 64, 65]
MAX_REF_M = 118  # largest reference block the Gibbs kernel's shared memory takes (test_plan_envelope.py pins it)
# accepted trees whose shapes reach the plan choices make_tree() leaves alone: name -> (levels, q, limited)
SHAPES = {
    # reference blocks of every tile-edge size (register and general factorisations), each with one leaf
    "ref_m_edges": ([[25], [EDGE_M + [MAX_REF_M]], [[4]] * (len(EDGE_M) + 1)], 1, False),
    # leaves of every tile-edge size up to a full work group, under one root: its staged rows take several chunks
    "leaf_m_edges": ([[25], [EDGE_M + [104, 105, 127, 128]]], 1, False),
    # parent sets of 15-17 and 31-33 rows (several roots), and of a few hundred rows
    "p_edges": ([[15, 16, 17, 31, 32, 33], [[7, 7]] * 6], 1, False),
    "p_hundreds": (chain(12, 30, 9), 1, False),
    "chain32": (chain(32, 5, 5), 1, False),
    "fanout": (_mixed_fanout(), 1, False),
    "fanout_q3": (_mixed_fanout(), 3, False),
    # all-NaN blocks (prediction blocks) among observed siblings, at a reference level and at the leaves
    "nan_siblings": ([[25], [[16, -9, 16, 16]], [[8, -8, 8], [], [-5], [8, 8]]], 3, False),
    "limited_fanout": (_mixed_fanout(), 1, True),
}


def shape_problem(name, seed=0):
    levels, q, limited = SHAPES[name]
    return make_shape_problem(levels, q=q, limited=limited, seed=seed)
