"""The search's network evaluator at every node of the tree, against the network and a float64 reference.

The evaluator after the tower (kv_mcts.cu: the heads, the legal-move logits that read only the policy_fc rows of the
legal moves, the softmax priors, the root noise and the value sign) runs in five kernels: mcts_eval_net_kernel, the split
pair mcts_head_kernel + mcts_eval_batch_kernel, mcts_late_net_kernel (cache hits and in-wave followers) and the two
root-mix kernels.  Here a real search runs with heads that pass the tower through (netref.live_heads), the oracle replays
it and lists every node's position, and every non-terminal node is compared with kv_net_forward on its position and
with the float64 graph:
  value            == +-kv_net_forward's value (side to move's view), bit for bit: the same device functions
  value            within 2e-2 of float64
  non-root priors  float64 softmax over kv_net_forward's logits of the legal moves, within 1e-6 + 1e-5 P (the kernels
                   sum the same 128 fp32 products in another order; on a B200 the largest error is 5e-8, a hundredth of
                   the bound); within 4e-2 of the float64 graph's softmax
  root priors      root_mix 0: (1 - eps) softmax + eps eta with the oracle's eta; root_mix 1: the reference rule on
                   kv_net_forward's 4096 logits; both within 1e-6 + 1e-5 P.  The reference rule is insensitive by nature
                   (softmax over 4096 logits, mixed with noise, renormalised): a root that got another position's softmax
                   statistics is off by only ~2e-5 with the reference net
  prior sums       1 within 1e-5
  terminal nodes   no edges, value -1 for checkmate and 0 otherwise, as the oracle's move generation says
"""
import time

import numpy as np
import pytest
import torch

import helpers as H
from knightvision_b200 import layout as L
from netref import Fp64Net, bnrand_net, live_heads, reference_rule_priors
from oracle import kv_oracle as O

pytestmark = pytest.mark.gpu

SIMS, SEED, GID, EPS, ALPHA, KMAX = 128, 17, 200, 0.25, 0.3, 8
VAL64, P64, PSUM = 2e-2, 4e-2, 1e-5
ARCHS = {"reference": dict(stem=256, tower=512, conv2=True, blocks=5),
         "256x2": dict(stem=256, tower=256, conv2=False, blocks=2)}
NET_SEED = {"reference": 31, "256x2": 32}    # fixed per architecture: a selection of tests builds the same networks
# (eval_split, cache log2, inflight K, root_mix, pipeline)
CONFIGS = ([(s, c, k, 0, 0) for s in (0, 1) for c in (0, 10, 18) for k in (1, 8)]
           + [(0, 0, 1, 1, 0), (0, 18, 8, 1, 0), (0, 10, 8, 0, 1)])


def _cfg_id(c):
    s, cache, k, rm, pipe = c
    return f"split{s}-cache{cache}-K{k}" + ("-rootmix" if rm else "") + ("-pipeline" if pipe else "")


def _tight(p):
    return 1e-6 + 1e-5 * p


def _bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)


def _softmax(x):
    e = np.exp(x - x.max())
    return e / e.sum()


def _move_index(mv):
    mv = mv.astype(np.int64)
    return (mv & 63) * 64 + ((mv >> 6) & 63)


@pytest.fixture(scope="module")
def eng():
    from knightvision_b200.engine import Engine
    e = Engine(0)
    yield e
    e.close()


@pytest.fixture(scope="module")
def roots():
    return H.search_roots()


_NETS = {}


def _net(arch):
    """(ChessNet, Fp64Net, memo of float64 outputs by position) per architecture, built once."""
    if arch not in _NETS:
        net = live_heads(bnrand_net(seed=NET_SEED[arch], **ARCHS[arch]))
        _NETS[arch] = (net, Fp64Net(net, "cuda"), {})
    return _NETS[arch]


def _fp64(ref, memo, lines, idx):
    """float64 (legal-move logits, value) of the graph for each line; memoised by line, since the configurations
    search the same trees."""
    keys = [l[:13].tobytes() for l in lines]
    todo = sorted({k: i for i, k in enumerate(keys) if k not in memo}.items(), key=lambda t: t[1])
    for c in range(0, len(todo), 512):
        part = [i for _, i in todo[c:c + 512]]
        x = torch.from_numpy(O.encode(lines[part])).cuda()
        with torch.no_grad():
            p, v = ref.forward(x)
        p, v = p.cpu().numpy(), v[:, 0].cpu().numpy()
        for j, i in enumerate(part):
            memo[keys[i]] = (p[j, idx[i]], float(v[j]))
    return [memo[k] for k in keys]


def _run(eng, G, K):
    if K == 1:
        eng.mcts_run_sims(SIMS)
        return
    eng.mcts_run_sims(1 + (SIMS - 1 + K - 1) // K)
    for _ in range(SIMS):
        if eng.mcts_status()["sims_in_move"] >= G * SIMS:
            return
        eng.mcts_run_sims(1)


@pytest.mark.parametrize("cfg", CONFIGS, ids=_cfg_id)
@pytest.mark.parametrize("arch", list(ARCHS))
def test_search_evaluator_every_node(eng, roots, arch, cfg, capsys):
    from knightvision_b200.engine import lines_to_device
    t0 = time.perf_counter()
    split, cache, K, root_mix, pipe = cfg
    lines, names = roots
    G = len(lines)
    net, ref, memo = _net(arch)
    net.attach(eng, max_batch=G * KMAX)
    eng.mcts_create(G, SIMS, max_plies=4, temp_plies=0, seed=SEED, eval_mode=1, inflight=K)
    try:
        eng.mcts_set_eval_split(split)
        eng.mcts_set_pipeline(pipe)
        eng.mcts_set_root_mix(root_mix)
        eng.mcts_enable_cache(cache)
        eng.mcts_reset(lines_to_device(lines, eng.device), game_id_base=GID)
        _run(eng, G, K)
        st = eng.mcts_status()
        dumps = [(eng.mcts_read_root(g),) + eng.mcts_dump_tree(g) for g in range(G)]
    finally:
        eng.mcts_enable_cache(0)
        eng.mcts_set_eval_split(-1)
        eng.mcts_set_pipeline(-1)
        eng.mcts_set_root_mix(-1)
    what = f"{arch} {_cfg_id(cfg)}"
    assert st["sims_in_move"] == G * SIMS and st["overflow"] == 0, (what, st)
    if cache:
        assert st["cache_hits"] > 0, what

    # the oracle replays each game's tree (the device's values and priors) and lists its nodes
    ocfg = O.mcts_cfg(SIMS, seed=SEED, inflight=K, root_mix=root_mix)
    nodes = []          # (game, node, depth, line, device value, device priors, move words)
    n_term = n_rewritten = 0
    for g, (got, nv, nf, ep, root) in enumerate(dumps):
        assert np.array_equal(root[:13], lines[g][:13]), (what, names[g])
        r = O.mcts_search(ocfg, root, game_id=GID + g, ply=0, replay=(nv, nf, ep), nodes=True)
        assert got["nodes"] == r["nodes"] and got["edges"] == r["edges"] and r["overflow"] == 0, (what, names[g])
        assert np.array_equal(got["N"], r["N"]) and np.array_equal(_bits(got["W"]), _bits(r["W"])), (what, names[g])
        nn = r["nodes"]
        assert np.array_equal(nf[:nn], r["node_first"]), (what, names[g], "node numbering")
        _, counts, flags, _ = O.movegen(r["node_line"].copy())
        term = (counts == 0) | ((flags & L.RF_ONLY_KINGS) != 0)
        assert np.array_equal(term, r["node_term"]), (what, names[g])
        exp_term = np.where((counts == 0) & ((flags & L.RF_CHECKMATE) != 0), -1.0, 0.0).astype(np.float32)
        assert np.array_equal(nv[:nn][term], exp_term[term]) and (nf[:nn][term] == -1).all(), (what, names[g], "terminal")
        n_term += int(term.sum())
        n_rewritten += int(not np.array_equal(r["node_line"][0], root))    # root evaluated after the movegen rewrite
        depth = np.zeros(nn, np.int64)
        for i in np.nonzero(~term)[0]:
            f, n = r["node_first"][i], r["node_n"][i]
            assert n == counts[i], (what, names[g], i)
            kids = r["edge_child"][f:f + n]
            depth[kids[kids >= 0]] = depth[i] + 1
            nodes.append((g, i, depth[i], r["node_line"][i], nv[i], ep[f:f + n], r["edge_mv"][f:f + n]))

    M = len(nodes)
    nl = np.stack([x[3] for x in nodes])
    wtm = (nl[:, 12] & np.uint64(1)).astype(bool)
    dep = np.array([x[2] for x in nodes])
    idx = [_move_index(x[6]) for x in nodes]
    pol, val = [], []
    for c in range(0, M, net.max_batch):
        p, v = net.forward_lines(torch.from_numpy(nl[c:c + net.max_batch].view(np.int64)).to(eng.device))
        pol.append(p.cpu().numpy())
        val.append(v[:, 0].cpu().numpy())
    pol, val = np.concatenate(pol), np.concatenate(val)
    ref64 = _fp64(ref, memo, nl, idx)

    # per node errors
    v_dev = np.array([x[4] for x in nodes], np.float32)
    v_net = np.where(wtm, val, -val).astype(np.float32)
    v_64 = np.where(wtm, 1.0, -1.0) * np.array([r[1] for r in ref64])
    val_mismatch = int((_bits(v_dev) != _bits(v_net)).sum())
    err = dict(val64=float(np.abs(v_dev - v_64).max()), nonroot=0.0, nonroot_r=0.0, root=0.0, root_r=0.0, psum=0.0,
               nonroot64=0.0)
    for j, (g, i, _, _, _, P, mv) in enumerate(nodes):
        P = P.astype(np.float64)
        err["psum"] = max(err["psum"], abs(P.sum() - 1.0))
        sm = _softmax(pol[j, idx[j]].astype(np.float64))
        if i == 0:
            if root_mix:
                want = reference_rule_priors(pol[j], mv, ALPHA, EPS, SEED, GID + g, 0)
            else:
                want = (1 - EPS) * sm + EPS * O.root_eta(ALPHA, SEED, GID + g, 0, len(mv)).astype(np.float64)
            e = np.abs(P - want)
            err["root"], err["root_r"] = max(err["root"], e.max()), max(err["root_r"], (e / _tight(want)).max())
        else:
            e = np.abs(P - sm)
            err["nonroot"], err["nonroot_r"] = max(err["nonroot"], e.max()), max(err["nonroot_r"], (e / _tight(sm)).max())
            err["nonroot64"] = max(err["nonroot64"], np.abs(P - _softmax(ref64[j][0])).max())
    # the heads are live: values and logits depend on the position, not on the policy_fc bias alone
    bias = net.policy_fc.bias.detach().cpu().numpy()
    v_std = float(v_net.std())
    lg_spread = max(float(np.abs(pol[j, idx[j]] - bias[idx[j]]).max()) for j in range(M))
    deep_w, deep_b = int(((dep >= 2) & wtm).sum()), int(((dep >= 2) & ~wtm).sum())
    kinds = np.bitwise_or.reduce(np.concatenate([x[6] >> 12 for x in nodes]))
    widest = max(len(x[6]) for x in nodes)
    with capsys.disabled():
        print(f"\n[{what}] {M} evaluated nodes ({deep_w} / {deep_b} at depth >= 2 with white / black to move), "
              f"{n_term} terminal, widest {widest} edges, {st['evals']} tower evaluations, {st['cache_hits']} cache hits; "
              f"value std {v_std:.3f}, max |logit - bias| {lg_spread:.3f}; {time.perf_counter() - t0:.1f} s\n"
              f"  value vs kv_net_forward: {val_mismatch} differing bits (bound 0); vs float64 max {err['val64']:.2e} "
              f"(bound {VAL64:.0e})\n"
              f"  non-root priors vs kv_net_forward softmax max {err['nonroot']:.2e} ({err['nonroot_r']:.3f} of "
              f"1e-6 + 1e-5 P); vs float64 max {err['nonroot64']:.2e} (bound {P64:.0e})\n"
              f"  root priors ({'reference rule' if root_mix else 'softmax + eps eta'}) max {err['root']:.2e} "
              f"({err['root_r']:.3f} of 1e-6 + 1e-5 P); prior sums max |sum - 1| {err['psum']:.2e} (bound {PSUM:.0e})")
    assert val_mismatch == 0, what
    assert err["val64"] <= VAL64, (what, err)
    assert err["nonroot_r"] <= 1.0 and err["root_r"] <= 1.0, (what, err)
    assert err["nonroot64"] <= P64 and err["psum"] <= PSUM, (what, err)
    # coverage: the comparisons above are not vacuous
    assert deep_w >= 100 and deep_b >= 100, what
    assert n_rewritten >= 1, what
    assert widest >= 100 and (kinds & (L.MF_EP | L.MF_CASTLE | L.MF_PROMO)) == 7, what
    assert v_std > 1e-2 and lg_spread > 0.1, (what, v_std, lg_spread)
