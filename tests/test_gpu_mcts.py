"""GPU tree search vs the sequential MCTS oracle.  Bit-exact visit counts / W / priors / chosen moves:
 - hash evaluator: the whole pipeline including softmax and Dirichlet arithmetic;
 - network evaluator: the oracle replays the values and priors the device recorded ("given identical net outputs")."""
import numpy as np
import pytest
import torch

import helpers as H
from netref import reference_rule_priors
from knightvision_b200 import layout as L
from oracle import kv_oracle as O

pytestmark = pytest.mark.gpu


def _bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)


@pytest.fixture(scope="module")
def eng():
    from knightvision_b200.engine import Engine
    e = Engine(0)
    yield e
    e.close()


def test_search_hash_evaluator_bit_exact(eng):
    from knightvision_b200.engine import lines_to_device
    lines = H.random_playout_positions(n_games=8, max_plies=120, seed=33)
    roots = lines[np.random.default_rng(1).permutation(len(lines))[:96]]
    roots[0] = L.start_line()
    sims = 200
    eng.mcts_create(len(roots), sims, max_plies=4, temp_plies=0, seed=77, eval_mode=0)
    eng.mcts_reset(lines_to_device(roots, eng.device), game_id_base=1000)
    eng.mcts_run_sims(sims)
    cfg = O.mcts_cfg(sims, seed=77)
    for g in range(len(roots)):
        got = eng.mcts_read_root(g)
        r = O.mcts_search(cfg, roots[g], game_id=1000 + g, ply=0)
        assert got["nodes"] == r["nodes"] and got["edges"] == r["edges"], g
        assert np.array_equal(got["moves"], r["moves"]) and np.array_equal(got["N"], r["N"]), g
        assert np.array_equal(_bits(got["W"]), _bits(r["W"])) and np.array_equal(_bits(got["P"]), _bits(r["P"])), g


def test_selfplay_games_hash_evaluator_bit_exact(eng):
    G, sims, max_plies = 48, 32, 60
    eng.mcts_create(G, sims, max_plies=max_plies, temp_plies=8, seed=5, eval_mode=0)
    eng.mcts_reset(None, game_id_base=0)
    for _ in range(max_plies):
        eng.mcts_run_move()
    st = eng.mcts_status()
    assert st["done"] == G and st["overflow"] == 0
    lines, move, reward, game = (t.cpu().numpy() for t in eng.mcts_records())
    lines = lines.view(np.uint64)
    cfg = O.mcts_cfg(sims, temp_plies=8, max_plies=max_plies, seed=5)
    total = 0
    for g in range(G):
        m, pos, res = O.selfplay_game(cfg, L.start_line(), game_id=g)
        sel = game == g
        assert sel.sum() == len(m), g
        assert np.array_equal(move[sel], [O.lib().kvo_move_index(int(x)) for x in m]), g
        assert np.array_equal(lines[sel][:, :12], pos[:, :12]), g
        exp_reward = 1.0 if res > 0 else (-1.0 if res < 0 else 0.2)
        assert np.allclose(reward[sel], exp_reward), g
        total += len(m)
    assert total == len(move) == st["plies"]


def test_search_with_network_replayed_by_oracle(eng):
    """Real tower + heads on the device; the oracle re-runs the search with the recorded values / priors."""
    from knightvision_b200.model import ChessNet
    torch.manual_seed(0)
    net = ChessNet().eval().attach(eng, max_batch=64)
    G, sims = 24, 160
    eng.mcts_create(G, sims, max_plies=8, temp_plies=0, seed=9, eval_mode=1)
    eng.mcts_reset(None, game_id_base=0)
    eng.mcts_run_sims(sims)
    cfg = O.mcts_cfg(sims, seed=9)
    for g in (0, 5, 23):
        got = eng.mcts_read_root(g)
        nv, nf, ep, root = eng.mcts_dump_tree(g)
        r = O.mcts_search(cfg, root, game_id=g, ply=0, replay=(nv, nf, ep))
        assert got["nodes"] == r["nodes"] and np.array_equal(got["N"], r["N"]), g
        assert np.array_equal(_bits(got["W"]), _bits(r["W"])), g
        assert int(got["N"].sum()) == sims - 1
        # priors are a softmax over the legal moves of the net's logits (masked softmax fused with the heads)
        pol, val = net.forward_lines(torch.from_numpy(root.view(np.int64)[None]).to(eng.device))
        idx = [O.lib().kvo_move_index(int(x)) for x in got["moves"]]
        lg = pol[0, idx].double().cpu().numpy()
        sm = np.exp(lg - lg.max()); sm /= sm.sum()
        # root priors carry Dirichlet noise: (1-eps) * softmax + eps * eta, eta >= 0, sum eta = 1
        eta = (got["P"].astype(np.float64) - 0.75 * sm) / 0.25
        assert eta.min() > -1e-4 and abs(eta.sum() - 1.0) < 1e-3
    # and play two moves so finish_move / tree reset are exercised with the net
    eng.mcts_finish_move()
    eng.mcts_run_move()
    st = eng.mcts_status()
    assert st["plies"] == 2 * G and st["evals"] > 0


def test_dropin_self_play_record_format(eng, monkeypatch):
    from knightvision_b200 import selfplay as SP
    from knightvision_b200.model import ChessNet
    monkeypatch.setattr(SP, "DEFAULT_SIMS", 16)
    monkeypatch.setitem(SP._engines, 0, eng)
    torch.manual_seed(1)
    data = SP.self_play(ChessNet().eval(), 3, torch.device("cuda:0"), max_moves=6)
    assert len(data) == 18
    s, mv, rw = data[0]
    assert isinstance(s, np.ndarray) and s.dtype == np.float32 and s.shape == (12, 8, 8)
    assert np.array_equal(s, O.encode(L.start_line()[None])[0])        # first record = initial position planes
    assert isinstance(mv, int) and 0 <= mv < 4096 and isinstance(rw, float) and rw == pytest.approx(0.2)
    assert SP.generate_self_play_data(ChessNet().eval(), 2, torch.device("cuda:0"), max_moves=4) is not None
    with pytest.raises(ValueError):
        SP.self_play(None, 1, torch.device("cuda:0"))
    with pytest.raises(FileNotFoundError):
        SP.self_play(None, 1, torch.device("cuda:0"), model_path="/nonexistent/model.pth")


def test_bench_dump_outputs(eng, tmp_path, monkeypatch):
    """bench.py --dump-outputs: float arrays that hold the roots exactly and the records as SelfPlay.records returns them;
    beyond DUMP_RECORDS records, every record of a fixed sample of games, the same on every call."""
    import bench_mcts as B
    from knightvision_b200.selfplay import records_to_tuples
    G, moves = 40, 5
    eng.mcts_create(G, 16, max_plies=30, temp_plies=4, seed=11, eval_mode=0)
    eng.mcts_reset(None, game_id_base=0)
    for _ in range(moves):
        eng.mcts_run_move()
    B.save_outputs(str(tmp_path), B.collect_outputs(eng, moves))
    got = {p.stem: np.load(p) for p in tmp_path.glob("*.npy")}
    assert sorted(got) == ["counters", "games", "record_game", "record_move", "record_planes", "record_reward", "roots"]
    assert all(a.dtype in (np.float32, np.float64) for a in got.values())
    assert got["games"].tolist() == list(range(G))
    roots = got["roots"].astype(np.uint16).view(np.int64)
    assert np.array_equal(roots, eng.mcts_roots().cpu().numpy())
    st = eng.mcts_status()
    assert got["counters"].tolist() == [st["done"], st["plies"], st["overflow"], st["white_wins"], st["black_wins"], st["draws"]]
    lines, move, reward, game = eng.mcts_records()
    recs = records_to_tuples(eng, lines, move, reward)
    assert len(recs) == st["plies"] > 64
    assert np.array_equal(got["record_planes"], np.stack([r[0] for r in recs]))
    assert got["record_move"].tolist() == [r[1] for r in recs] and got["record_reward"].tolist() == [r[2] for r in recs]
    assert np.array_equal(got["record_game"], game.cpu().numpy())

    monkeypatch.setattr(B, "DUMP_RECORDS", 64)
    a, b = B.collect_outputs(eng, moves), B.collect_outputs(eng, moves)
    games = B.dump_games(G, moves)
    assert len(games) == 64 // moves and np.array_equal(a["games"], games)
    keep = np.isin(got["record_game"], games)
    assert len(a["record_game"]) <= 64 and set(a["record_game"].tolist()) == set(games.tolist())
    for name in ("record_planes", "record_move", "record_reward", "record_game"):
        assert np.array_equal(a[name], got[name][keep]) and np.array_equal(a[name], b[name]), name
    assert np.array_equal(a["roots"], got["roots"][games])


def test_full_size_wave_4096_games(eng):
    """BASELINE config 3 size: 4 096 concurrent games; size-independent invariants after 12 waves."""
    from knightvision_b200.model import ChessNet
    torch.manual_seed(0)
    ChessNet().eval().attach(eng, max_batch=4096)
    eng.mcts_create(4096, 12, max_plies=4, temp_plies=0, seed=3, eval_mode=1)
    eng.mcts_reset(None, 0)
    eng.mcts_run_sims(12)
    st = eng.mcts_status()
    assert st["sims_in_move"] == 4096 * 12 and st["evals"] == 4096 * 12   # no terminal leaf this early
    r0, r1 = eng.mcts_read_root(0), eng.mcts_read_root(4095)
    assert int(r0["N"].sum()) == 11 and int(r1["N"].sum()) == 11 and len(r0["moves"]) == 20
    eng.mcts_finish_move()
    assert eng.mcts_status()["plies"] == 4096


def _play_records(eng, G, sims, moves, eval_mode, cache_log2, seed=13, pipeline=0, inflight=1):
    eng.mcts_create(G, sims, max_plies=moves, temp_plies=4, seed=seed, eval_mode=eval_mode, inflight=inflight)
    eng.mcts_set_pipeline(pipeline)
    eng.mcts_enable_cache(cache_log2)
    eng.mcts_reset(None, game_id_base=50)
    roots = []
    for i in range(moves):
        if inflight == 1:
            eng.mcts_run_sims(sims)
        else:
            eng.mcts_run_sims(1 + (sims - 2 + inflight) // inflight)
            while True:
                st = eng.mcts_status()
                if st["sims_in_move"] >= (G - st["done"]) * sims:
                    break
                eng.mcts_run_sims(1)
        if i == moves - 1:
            roots = [eng.mcts_read_root(g) for g in (0, G // 2, G - 1)]
        eng.mcts_finish_move()
    st = eng.mcts_status()
    rec = tuple(t.cpu().numpy() for t in eng.mcts_records())
    return rec, roots, st


@pytest.mark.parametrize("eval_mode", [0, 1])
def test_eval_cache_is_transparent(eng, eval_mode):
    """Same games, visit counts and W bits with the evaluation cache off, tiny (evictions) and roomy."""
    if eval_mode == 1:
        from knightvision_b200.model import ChessNet
        torch.manual_seed(0)
        ChessNet().eval().attach(eng, max_batch=256)
    G, sims, moves = 192, 40, 5
    base, broots, bst = _play_records(eng, G, sims, moves, eval_mode, 0)
    assert bst["cache_hits"] == 0 and bst["evals"] > 0
    for log2 in (10, 18):
        rec, roots, st = _play_records(eng, G, sims, moves, eval_mode, log2)
        for a, b in zip(base, rec):
            assert np.array_equal(a, b)
        for ra, rb in zip(broots, roots):
            assert np.array_equal(ra["N"], rb["N"]) and np.array_equal(_bits(ra["W"]), _bits(rb["W"]))
            assert np.array_equal(_bits(ra["P"]), _bits(rb["P"]))
        assert st["cache_hits"] > 0 and st["evals"] + st["cache_hits"] == bst["evals"]
    eng.mcts_enable_cache(0)


@pytest.mark.parametrize("eval_mode,K", [(0, 1), (1, 1), (1, 4)])
def test_pipelined_groups_are_transparent(eng, eval_mode, K):
    """Two game groups whose waves alternate on two streams (kv_mcts_set_pipeline): the same games, visit counts, W and
    prior bits as the single-stream schedule, with the shared evaluation cache off, tiny (evictions while the other
    group's evaluator is filling) and roomy (leaves of one group following leaders of the other)."""
    if eval_mode == 1:
        from knightvision_b200.model import ChessNet
        torch.manual_seed(0)
        ChessNet().eval().attach(eng, max_batch=200 * K)
    G, sims, moves = 200, 40, 5          # groups of 104 + 96 games
    base, broots, bst = _play_records(eng, G, sims, moves, eval_mode, 0, pipeline=0, inflight=K)
    for log2 in (0, 10, 18):
        rec, roots, st = _play_records(eng, G, sims, moves, eval_mode, log2, pipeline=1, inflight=K)
        for a, b in zip(base, rec):
            assert np.array_equal(a, b)
        for ra, rb in zip(broots, roots):
            assert np.array_equal(ra["N"], rb["N"]) and np.array_equal(_bits(ra["W"]), _bits(rb["W"]))
            assert np.array_equal(_bits(ra["P"]), _bits(rb["P"]))
        assert st["evals"] + st["cache_hits"] == bst["evals"] and (st["cache_hits"] > 0) == (log2 > 0)
    eng.mcts_enable_cache(0)


def test_pipelined_selfplay_hash_evaluator_matches_oracle(eng):
    """Whole games through kv_mcts_run_move with the pipelined schedule, against the sequential oracle."""
    G, sims, max_plies = 40, 24, 30
    eng.mcts_create(G, sims, max_plies=max_plies, temp_plies=8, seed=15, eval_mode=0)
    eng.mcts_set_pipeline(1)
    eng.mcts_enable_cache(12)
    eng.mcts_reset(None, game_id_base=0)
    for _ in range(max_plies):
        eng.mcts_run_move()
    st = eng.mcts_status()
    assert st["done"] == G and st["cache_hits"] > 0
    rl, move, reward, game = (t.cpu().numpy() for t in eng.mcts_records())
    cfg = O.mcts_cfg(sims, temp_plies=8, max_plies=max_plies, seed=15)
    for g in range(G):
        m, pos, res = O.selfplay_game(cfg, L.start_line(), game_id=g)
        sel = game == g
        assert sel.sum() == len(m), g
        assert np.array_equal(move[sel], [O.lib().kvo_move_index(int(x)) for x in m]), g
        assert np.array_equal(rl.view(np.uint64)[sel][:, :12], pos[:, :12]), g
    eng.mcts_enable_cache(0)


def test_learn_loop_small_tower(eng, monkeypatch):
    """scripts/learn.py loop semantics on a small tower: train -> self-play -> extend; the engine picks up the
    trained weights (and drops the evaluation cache) between iterations."""
    from knightvision_b200 import learn as LR
    from knightvision_b200 import selfplay as SP
    from knightvision_b200.model import ChessNet
    monkeypatch.setitem(SP._engines, 0, eng)
    torch.manual_seed(3)
    net = ChessNet(stem=64, tower=256, blocks=1, conv2=True, max_batch=32)
    cfg = LR.build_cfg(num_iterations=2, device=torch.device("cuda:0"))
    cfg.selfplay.num_games, cfg.selfplay.max_moves, cfg.selfplay.sims = 16, 6, 12
    cfg.train.epochs, cfg.train.batch_size = 1, 32
    before = net.weight_blob().clone()
    net, data, hist = LR.reinforcement_loop(cfg, net=net)
    assert len(hist) == 2 and hist[0]["records"] == 16 * 6 and len(data) == 2 * 16 * 6
    assert np.isnan(hist[0]["loss"]) and np.isfinite(hist[1]["loss"])     # nothing to train on before the first games
    assert not torch.equal(before, net.weight_blob())
    # reference-format records round-trip through the packed store
    d2 = LR.ReplayData(eng)
    d2.extend([(O.encode(L.start_line()[None])[0], 3364, 0.2)])
    assert int(d2.move[0]) == 3364 and np.array_equal(d2.lines[0, :12].cpu().numpy().view(np.uint64), L.start_line()[:12])


@pytest.mark.parametrize("K", [4, 16])
def test_virtual_loss_inflight_hash_evaluator_bit_exact(eng, K):
    """K simulations in flight per game and wave with virtual loss (SURVEY 8a row M3): whole games, bit-exact with the
    oracle's wave emulation — visit counts, W bits, priors, chosen moves, records."""
    from knightvision_b200.engine import lines_to_device
    lines = H.random_playout_positions(n_games=8, max_plies=120, seed=35)
    roots = lines[np.random.default_rng(2).permutation(len(lines))[:64]]
    roots[0] = L.start_line()
    sims = 200
    eng.mcts_create(len(roots), sims, max_plies=4, temp_plies=0, seed=78, eval_mode=0, inflight=K)
    eng.mcts_enable_cache(12 if K == 16 else 0)        # the cache stays transparent with several leaves per game
    eng.mcts_reset(lines_to_device(roots, eng.device), game_id_base=500)
    w0 = eng.mcts_waves()
    eng.mcts_run_sims(1 + (sims - 1 + K - 1) // K)      # the minimum; collisions may leave some simulations to run
    left = len(roots) * sims - eng.mcts_status()["sims_in_move"]
    while left:
        eng.mcts_run_sims(1)
        left = len(roots) * sims - eng.mcts_status()["sims_in_move"]
    assert eng.mcts_waves() - w0 < sims                  # far fewer waves than simulations
    cfg = O.mcts_cfg(sims, seed=78, inflight=K)
    for g in range(len(roots)):
        got = eng.mcts_read_root(g)
        r = O.mcts_search(cfg, roots[g], game_id=500 + g, ply=0)
        assert got["nodes"] == r["nodes"] and got["edges"] == r["edges"], g
        assert np.array_equal(got["moves"], r["moves"]) and np.array_equal(got["N"], r["N"]), g
        assert np.array_equal(_bits(got["W"]), _bits(r["W"])) and np.array_equal(_bits(got["P"]), _bits(r["P"])), g
        if len(r["N"]):
            assert int(got["N"].sum()) == sims - 1
    eng.mcts_enable_cache(0)
    # whole games through kv_mcts_run_move (its own wave loop)
    G, sims, max_plies = 32, 48, 40
    eng.mcts_create(G, sims, max_plies=max_plies, temp_plies=8, seed=6, eval_mode=0, inflight=K)
    eng.mcts_reset(None, game_id_base=0)
    for _ in range(max_plies):
        eng.mcts_run_move()
    st = eng.mcts_status()
    assert st["done"] == G and st["overflow"] == 0
    rl, move, reward, game = (t.cpu().numpy() for t in eng.mcts_records())
    cfg = O.mcts_cfg(sims, temp_plies=8, max_plies=max_plies, seed=6, inflight=K)
    for g in range(G):
        m, pos, res = O.selfplay_game(cfg, L.start_line(), game_id=g)
        sel = game == g
        assert sel.sum() == len(m), g
        assert np.array_equal(move[sel], [O.lib().kvo_move_index(int(x)) for x in m]), g
        assert np.array_equal(rl.view(np.uint64)[sel][:, :12], pos[:, :12]), g


def test_virtual_loss_inflight_with_network_replayed_by_oracle(eng):
    """512 leaves per wave from 64 games x 8 in flight through the real tower; the oracle replays the recorded values
    and priors through its own wave emulation."""
    from knightvision_b200.model import ChessNet
    torch.manual_seed(0)
    ChessNet().eval().attach(eng, max_batch=512)
    G, sims, K = 64, 160, 8
    eng.mcts_create(G, sims, max_plies=8, temp_plies=0, seed=9, eval_mode=1, inflight=K)
    for cache in (0, 14):
        eng.mcts_enable_cache(cache)
        eng.mcts_reset(None, game_id_base=0)
        eng.mcts_run_sims(1 + (sims - 1 + K - 1) // K)
        while eng.mcts_status()["sims_in_move"] < G * sims:
            eng.mcts_run_sims(1)
        cfg = O.mcts_cfg(sims, seed=9, inflight=K)
        for g in (0, 31, 63):
            got = eng.mcts_read_root(g)
            nv, nf, ep, root = eng.mcts_dump_tree(g)
            r = O.mcts_search(cfg, root, game_id=g, ply=0, replay=(nv, nf, ep))
            assert got["nodes"] == r["nodes"] and np.array_equal(got["N"], r["N"]), g
            assert np.array_equal(_bits(got["W"]), _bits(r["W"])), g
            assert int(got["N"].sum()) == sims - 1
        st = eng.mcts_status()
        assert st["evals"] + st["cache_hits"] <= G * sims and st["evals"] > 0
    eng.mcts_enable_cache(0)
    eng.mcts_reset(None, game_id_base=0)
    eng.mcts_run_move()
    eng.mcts_run_move()
    assert eng.mcts_status()["plies"] == 2 * G


def test_evaluation_players(eng, monkeypatch):
    """scripts/play_vs_model.py:34-49 greedy player, the single-position search player (virtual loss fills the batch) and
    the two-network arena."""
    from knightvision_b200 import chess_engine as CE
    from knightvision_b200 import players as P
    from knightvision_b200 import selfplay as SP
    from knightvision_b200.ai import encode_board, encode_move
    from knightvision_b200.model import ChessNet
    monkeypatch.setitem(SP._engines, 0, eng)
    CE.set_engine(eng)
    torch.manual_seed(2)
    net = ChessNet().eval()
    gs = CE.GameState()
    mv = P.get_ai_move(gs, net)
    legal = gs.getValidMoves()
    assert mv in legal
    pol, _ = net(torch.from_numpy(encode_board(gs.board)[None]).cuda())
    idx = [encode_move(m.startRow, m.startCol, m.endRow, m.endCol) for m in legal]
    assert mv == legal[int(np.argmax(pol[0, idx].cpu().numpy()))]           # masked argmax of the policy
    # mate in one (several mating moves exist): kings + white queen, white to move
    gs = CE.GameState()
    gs.board = [["--"] * 8 for _ in range(8)]
    gs.board[0][7], gs.board[2][6], gs.board[1][0] = "bK", "wK", "wQ"
    gs.blackKingLocation, gs.whiteKingLocation = (0, 7), (2, 6)
    gs.wKingMoved = gs.bKingMoved = True
    gs.whiteToMove = True
    m = P.get_mcts_move(gs, net, sims=600, inflight=16, engine=eng)
    assert m in gs.getValidMoves()
    gs.makeMove(m)
    assert gs.getValidMoves() == [] and gs.checkMate
    # arena: every game is accounted for
    torch.manual_seed(3)
    other = ChessNet().eval()
    r = P.arena(net, other, n_games=8, sims=8, max_plies=6, device="cuda:0")
    assert r["a_wins"] + r["b_wins"] + r["draws"] == 8 and r["games"] == 8


def test_reference_rule_mode_hash_evaluator_bit_exact(eng):
    """sims = 1: no search, the move is sampled from root priors mixed the reference's way (softmax and Dirichlet noise
    over all 4096 indices, scripts/self_play.py:150-167), resignation on.  Whole games and priors bit-exact vs the oracle."""
    G, max_plies = 96, 48
    eng.mcts_create(G, 1, max_plies=max_plies, temp_plies=0, seed=21, eval_mode=0)
    eng.mcts_reset(None, game_id_base=300)
    eng.mcts_run_sims(1)
    cfg = O.mcts_cfg(1, max_plies=max_plies, seed=21)
    for g in (0, 41, 95):
        got = eng.mcts_read_root(g)
        r = O.mcts_search(cfg, L.start_line(), game_id=300 + g, ply=0)
        assert np.array_equal(got["moves"], r["moves"]) and np.array_equal(_bits(got["P"]), _bits(r["P"])), g
        lg, _ = O.hash_eval(L.start_line())
        assert np.allclose(got["P"], reference_rule_priors(lg, got["moves"], 0.3, 0.25, 21, 300 + g, 0), rtol=2e-5)
    eng.mcts_finish_move()
    for _ in range(max_plies):
        eng.mcts_run_move()
    st = eng.mcts_status()
    assert st["done"] == G
    lines, move, reward, game = (t.cpu().numpy() for t in eng.mcts_records())
    lines = lines.view(np.uint64)
    resigned = 0
    for g in range(G):
        m, pos, res = O.selfplay_game(cfg, L.start_line(), game_id=300 + g)
        sel = game == g
        assert sel.sum() == len(m), g
        assert np.array_equal(move[sel], [O.lib().kvo_move_index(int(x)) for x in m]), g
        assert np.array_equal(lines[sel][:, :12], pos[:, :12]), g
        assert np.allclose(reward[sel], 1.0 if res > 0 else (-1.0 if res < 0 else 0.2)), g
        resigned += int(len(m) < max_plies and res != 0)
    assert resigned > G // 2          # hash values below -0.7 come up within a few plies after move 15


def test_reference_rule_mode_network_priors(eng):
    """Same mode with the real network: the root priors follow the reference's formula on the net's own logits, for a
    tower evaluation, an in-wave follower and a cache hit alike."""
    from knightvision_b200.model import ChessNet
    torch.manual_seed(0)
    net = ChessNet().eval().attach(eng, max_batch=64)
    G = 12
    eng.mcts_create(G, 1, max_plies=6, temp_plies=0, seed=8, eval_mode=1)
    eng.mcts_enable_cache(12)
    eng.mcts_reset(None, game_id_base=70)
    eng.mcts_run_sims(1)
    st = eng.mcts_status()
    assert st["evals"] >= 1 and st["evals"] + st["cache_hits"] == G   # leaders (tower) + followers of the same wave
    pol, val = net.forward_lines(torch.from_numpy(L.start_line().view(np.int64)[None]).to(eng.device))
    lg = pol[0].float().cpu().numpy()
    first = {}
    for g in (0, 5, 11):
        got = eng.mcts_read_root(g)
        want = reference_rule_priors(lg, got["moves"], 0.3, 0.25, 8, 70 + g, 0)
        assert np.allclose(got["P"], want, rtol=1e-3, atol=1e-6), g
        first[g] = got["P"].copy()
    # the same roots again, now served by the cache (late kernel): identical bits
    eng.mcts_reset(None, game_id_base=70)
    eng.mcts_run_sims(1)
    st2 = eng.mcts_status()
    assert st2["evals"] == 0 and st2["cache_hits"] == G
    for g in (0, 5, 11):
        assert np.array_equal(_bits(eng.mcts_read_root(g)["P"]), _bits(first[g])), g
    eng.mcts_finish_move()
    eng.mcts_run_move()                                               # ply 1: positions differ, hits from ply 0 do not apply
    roots = eng.mcts_roots().cpu().numpy().view(np.uint64)
    eng.mcts_run_sims(1)
    pol, _ = net.forward_lines(torch.from_numpy(roots.view(np.int64)).to(eng.device))
    for g in (1, 7):
        got = eng.mcts_read_root(g)
        want = reference_rule_priors(pol[g].float().cpu().numpy(), got["moves"], 0.3, 0.25, 8, 70 + g, 2)
        assert np.allclose(got["P"], want, rtol=1e-3, atol=1e-6), g
    eng.mcts_enable_cache(0)


def test_run_move_reports_exhausted_wave_budget(eng):
    """K > 1: kv_mcts_run_move returns an error instead of silently finishing a move that still owes simulations."""
    eng.mcts_create(4, 8, max_plies=4, temp_plies=0, seed=1, eval_mode=0, inflight=4)
    eng.mcts_reset(None, 0)
    eng.mcts_run_move()                 # the normal case completes
    assert eng.mcts_status()["plies"] == 4


def test_split_evaluator_matches_single_kernel(eng):
    """The two-kernel evaluator (head features, then eight leaves per CTA with a batched value MLP) gives the same games,
    visit counts, W and prior bits as the one-CTA-per-leaf kernel, with and without the evaluation cache."""
    from knightvision_b200.model import ChessNet
    torch.manual_seed(0)
    ChessNet().eval().attach(eng, max_batch=256)
    G, sims, moves = 173, 40, 4           # not a multiple of 8: a partly filled last CTA
    out = {}
    for split in (0, 1):
        for log2 in (0, 16):
            eng.mcts_create(G, sims, max_plies=moves, temp_plies=4, seed=13, eval_mode=1)
            eng.mcts_set_eval_split(split)
            eng.mcts_enable_cache(log2)
            eng.mcts_reset(None, game_id_base=50)
            for i in range(moves):
                eng.mcts_run_sims(sims)
                if i == moves - 1:
                    roots = [eng.mcts_read_root(g) for g in (0, G // 2, G - 1)]
                eng.mcts_finish_move()
            out[(split, log2)] = (tuple(t.cpu().numpy() for t in eng.mcts_records()), roots)
    base_rec, base_roots = out[(0, 0)]
    for key, (rec, roots) in out.items():
        for a, b in zip(base_rec, rec):
            assert np.array_equal(a, b), key
        for ra, rb in zip(base_roots, roots):
            assert np.array_equal(ra["N"], rb["N"]) and np.array_equal(_bits(ra["W"]), _bits(rb["W"])), key
            assert np.array_equal(_bits(ra["P"]), _bits(rb["P"])), key
    eng.mcts_enable_cache(0)
    eng.mcts_set_eval_split(-1)


def test_full_size_move_4096_games_800_sims_cache_transparent(eng):
    """BASELINE config 3 at full size: one move of 4 096 games x 800 simulations from random positions, with the
    evaluation cache and without it — the same moves for every game (argmax of the visit counts), every game played
    exactly one ply, no edge-pool overflow, and simulations = games x 800 on the device's counters."""
    from knightvision_b200.model import ChessNet
    torch.manual_seed(0)
    ChessNet().eval().attach(eng, max_batch=4096)
    G, sims = 4096, 800
    eng.mcts_create(G, sims, max_plies=8, temp_plies=0, seed=3, eval_mode=1)
    start = eng.random_positions(G, 40, 99)
    moves = {}
    for log2 in (22, 0):
        eng.mcts_enable_cache(log2)
        eng.mcts_reset(start, 0)
        eng.mcts_run_sims(sims)
        st = eng.mcts_status()
        assert st["sims_in_move"] == G * sims and st["overflow"] == 0
        assert st["evals"] + st["cache_hits"] <= G * sims and (st["cache_hits"] > 0) == (log2 > 0)
        r = eng.mcts_read_root(G - 1)
        assert int(r["N"].sum()) == sims - 1
        eng.mcts_finish_move()
        assert eng.mcts_status()["plies"] == G
        lines, move, reward, game = eng.mcts_records()
        assert game.cpu().tolist() == list(range(G))
        moves[log2] = move.cpu().numpy()
    assert np.array_equal(moves[22], moves[0])
    eng.mcts_enable_cache(0)
