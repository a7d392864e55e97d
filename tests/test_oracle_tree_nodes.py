"""The oracle's tree dump (O.mcts_search(..., nodes=True)): the tree the network-search tests replay and evaluate node by
node.  In hash mode every node and edge is re-derived from the rules and the hash evaluator; replay mode rebuilds the
same tree from the dumped values and priors."""
import numpy as np
import pytest

import helpers as H
from knightvision_b200 import layout as L
from oracle import kv_oracle as O

SEED, EPS, ALPHA = 23, 0.25, 0.3


def _bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)


def _expf(x):
    """include/kv_detmath.h kvd_expf in float32, one rounding per operation (no FMA), elementwise."""
    f = np.float32
    x = np.minimum(np.asarray(x, np.float32), f(88.0))
    t = x * f(1.44269504088896341)
    k = (t + np.where(t < 0, f(-0.5), f(0.5))).astype(np.int32)          # C cast: truncation toward zero
    kf = k.astype(np.float32)
    r = x - kf * f(0.693359375)
    r = r - kf * f(-2.12194440e-4)
    p = np.full_like(r, f(1.9875691500e-4))
    for c in (1.3981999507e-3, 8.3334519073e-3, 4.1665795894e-2, 1.6666665459e-1, 5.0000001201e-1):
        p = p * r + f(c)
    p = p * (r * r) + r
    p = p + f(1.0)
    out = p * ((k + 127).astype(np.uint32) << np.uint32(23)).view(np.float32)
    return np.where(np.asarray(x) < f(-87.0), f(0.0), out).astype(np.float32)


def _hash_priors(line, moves, root, game_id):
    """Priors of the hash evaluator by the legal-move rule (priors_from_logits), float32 in the oracle's order."""
    lg, _ = O.hash_eval(line)
    lg = lg[[O.lib().kvo_move_index(int(m)) for m in moves]]
    e = _expf(lg - lg.max())
    s = np.float32(0.0)
    for x in e:
        s = np.float32(s + x)
    p = e / s
    if root:
        p = np.float32(1.0 - EPS) * p + np.float32(EPS) * O.root_eta(ALPHA, SEED, game_id, 0, len(moves))
    return p.astype(np.float32)


def _check_tree(r, root_line, game_id, what):
    nn, ne = r["nodes"], r["edges"]
    nl, first, n = r["node_line"], r["node_first"], r["node_n"]
    assert r["overflow"] == 0 and nn > 1, what
    moves, counts, flags, after = O.movegen(nl.copy())
    assert np.array_equal(after, nl), what + ": a node line is not its own movegen result"
    # node 0 is the root as move generation leaves it
    assert np.array_equal(nl[0], O.movegen(root_line[None].copy())[3][0]), what
    assert np.array_equal(r["moves"], r["edge_mv"][first[0]:first[0] + n[0]]), what
    parent = np.full(nn, -1)
    for i in range(nn):
        term = (counts[i] == 0) or bool(flags[i] & L.RF_ONLY_KINGS)
        assert r["node_term"][i] == term, (what, i)
        if term:
            assert n[i] == 0 and first[i] == -1, (what, i)
            exp = -1.0 if (counts[i] == 0 and flags[i] & L.RF_CHECKMATE) else 0.0
            assert r["node_val"][i] == exp, (what, i)
            continue
        e = slice(first[i], first[i] + n[i])
        assert n[i] == counts[i] and np.array_equal(r["edge_mv"][e], moves[i, :n[i]]), (what, i, "edges != movegen")
        assert np.array_equal(_bits(r["edge_P"][e]), _bits(_hash_priors(nl[i], moves[i, :n[i]], i == 0, game_id))), \
            (what, i, "priors")
        _, v = O.hash_eval(nl[i])
        assert r["node_val"][i] == np.float32(v if int(nl[i][12]) & 1 else -v), (what, i)
        kids = r["edge_child"][e]
        assert int(r["edge_N"][e].sum()) + 1 == r["node_N"][i], (what, i)
        for k in np.nonzero(kids >= 0)[0]:
            c = kids[k]
            assert parent[c] == -1 and c > i, (what, c)
            parent[c] = i
            child = O.movegen(O.make_moves(nl[i][None], r["edge_mv"][first[i] + k][None]))[3][0]
            assert np.array_equal(nl[c], child), (what, i, c, "child line")
    assert (parent[1:] >= 0).all() and parent[0] == -1, what + ": every node but the root has one parent"
    assert (r["edge_child"] < nn).all()
    live = np.nonzero(~r["node_term"])[0]        # edge blocks tile the pool in creation order
    assert np.array_equal(first[live], np.concatenate([[0], np.cumsum(n[live])[:-1]])) and n[live].sum() == ne, what
    return nl


@pytest.mark.parametrize("K", [1, 8])
def test_tree_dump_hash_mode_and_replay(K):
    roots, names = H.search_roots()
    sims = 96
    cfg = O.mcts_cfg(sims, seed=SEED, inflight=K)
    seen_big = seen_rewrite = False
    for g, (root, name) in enumerate(zip(roots, names)):
        r = O.mcts_search(cfg, root, game_id=40 + g, ply=0, nodes=True)
        plain = O.mcts_search(cfg, root, game_id=40 + g, ply=0)
        for k in ("move", "nodes", "edges", "overflow"):
            assert r[k] == plain[k], (name, k)
        for k in ("moves", "N", "W", "P"):
            assert np.array_equal(_bits(r[k]) if r[k].dtype == np.float32 else r[k], _bits(plain[k]) if plain[k].dtype ==
                                  np.float32 else plain[k]), (name, k)
        _check_tree(r, root, 40 + g, name)
        seen_big |= int(r["node_n"].max()) >= 100
        seen_rewrite |= not np.array_equal(r["node_line"][0], root)
        # replay mode: the dumped values and priors, indexed by node as the device dumps them, rebuild the same tree
        nv = np.zeros(sims + 1, np.float32)
        nf = np.full(sims + 1, -1, np.int32)
        nv[:r["nodes"]], nf[:r["nodes"]] = r["node_val"], r["node_first"]
        rep = O.mcts_search(cfg, root, game_id=40 + g, ply=0, replay=(nv, nf, r["edge_P"]), nodes=True)
        for k in ("node_line", "node_first", "node_n", "node_N", "edge_mv", "edge_child", "edge_N"):
            assert np.array_equal(rep[k], r[k]), (name, k)
        for k in ("node_val", "edge_P", "edge_W"):
            assert np.array_equal(_bits(rep[k]), _bits(r[k])), (name, k)
    assert seen_big and seen_rewrite


def test_search_roots_cover_the_cases():
    roots, names = H.search_roots()
    moves, counts, flags, _ = O.movegen(roots.copy())
    assert (counts > 0).all() and not (flags & L.RF_ONLY_KINGS).any()
    wtm = (roots[:, 12] & np.uint64(1)).astype(bool)
    assert wtm.sum() >= 8 and (~wtm).sum() >= 8
    assert counts.max() >= 100
    assert ((flags & L.RF_STATE_MUTATED) != 0).sum() == 1       # the evaluated position is the rewritten line
    kinds = np.concatenate([moves[i, :counts[i]] >> 12 for i in range(len(roots))])
    for f in (L.MF_EP, L.MF_CASTLE, L.MF_PROMO):
        assert (kinds & f).any(), f
    # the three variants: same bitboards as another root, different legal moves
    for v in (-3, -2, -1):
        same = [i for i in range(len(roots) - 3) if np.array_equal(roots[i, :12], roots[v, :12])]
        assert same, names[v]
        for i in same:
            assert roots[i, 12] != roots[v, 12]
            assert counts[i] != counts[v] or not np.array_equal(moves[i], moves[v]), names[v]
