"""bench.py's self-play workload (BASELINE.json configs[2] / configs[3]): 4 096 concurrent games per GPU, 800 PUCT
simulations per move, the reference policy/value net (random init, torch.manual_seed(0), BN folded, bf16 tensor-core
tower), all games from the initial position.  One step = one move for every game = 800 search waves.
Games shard over ranks by game id (no data-path collective); NCCL only broadcasts the weight blob before the
generation and gathers the per-rank record counts after it.
"""
from __future__ import annotations

import json
import os
import time

import numpy as np

GAMES_PER_GPU = int(os.getenv("KV_BENCH_GAMES", "4096"))
SIMS = int(os.getenv("KV_BENCH_SIMS", "800"))
MAX_PLIES = 512
INFLIGHT = int(os.getenv("KV_BENCH_INFLIGHT", "8"))         # phase E: G/K games x K simulations in flight (0/1 = skip)
POLICY_MODE_PLIES = int(os.getenv("KV_BENCH_POLICY_PLIES", "40"))   # phase F: plies of reference-rule self-play (0 = skip)
CACHE_LOG2 = int(os.getenv("KV_BENCH_CACHE_LOG2", "24"))   # evaluation cache: 2^24 x 640 B = 10.7 GB (0 = off)
CONV_FLOPS_PER_EVAL = 2.0 * 64 * 9 * (256 * 512 + 10 * 512 * 512)      # conv2 + 5 residual blocks (tcgen05 kernel)
NET_FLOPS_PER_EVAL = 2.0 * 1587872256                                   # whole net, SURVEY §8d


def _ncu_traffic():
    """Average DRAM bytes (read + write) per launch of the tower kernel from the committed ncu capture, or None."""
    import glob
    import re
    root = os.path.dirname(os.path.abspath(__file__))
    files = sorted(glob.glob(os.path.join(root, "profiles", "*ncu_tower_umma2*.txt")))
    if not files:
        return None, None
    unit = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
    txt = open(files[-1]).read()
    rd = [float(v) * unit[u] for v, u in re.findall(r"dram__bytes_read\.sum\s+([0-9.]+) (\w*byte)", txt)]
    wr = [float(v) * unit[u] for v, u in re.findall(r"dram__bytes_write\.sum\s+([0-9.]+) (\w*byte)", txt)]
    if not rd or len(rd) != len(wr):
        return None, None
    return (sum(rd) + sum(wr)) / len(rd), os.path.relpath(files[-1], root)


CPU_GAMES = int(os.getenv("KV_BENCH_CPU_GAMES", "64"))


def random_start_lines(n, plies, seed):
    """n positions after `plies` uniformly random legal plies from the initial position (rules by the oracle)."""
    from knightvision_b200 import layout as L
    from oracle import kv_oracle as O
    rng = np.random.default_rng(seed)
    lines = np.stack([L.start_line()] * n)
    for _ in range(plies):
        moves, counts, flags, mid = O.movegen(lines.copy())
        pick = np.full(n, 0xFFFF, np.uint16)
        ok = (counts > 0) & ((flags & L.RF_ONLY_KINGS) == 0)
        idx = (rng.random(n) * np.maximum(counts, 1)).astype(np.int64)
        pick[ok] = moves[np.arange(n), idx][ok]
        lines = O.make_moves(mid, pick)
    lines[:, 13:] = 0
    return lines


class CpuSelfPlay:
    """The CPU implementation of the same path, run for real: CPU_GAMES games from the initial position searched in lock
    step by the sequential PUCT oracle (oracle/kv_oracle.c, step-wise API) — one simulation per game and wave, like the
    device engine — with the leaves of a wave evaluated as ONE batch by the reference network graph in fp32 on torch's CPU
    kernels, all host threads.  Like the device engine it evaluates a position only once (dictionary keyed by the 12
    bitboards, the network's whole input).  Same search constants, same weights (seed 0), same start."""

    def __init__(self, sims, n_games=CPU_GAMES, seed=42, start_lines=None):
        import torch
        from knightvision_b200 import layout as L
        from knightvision_b200.model import ChessNet
        from oracle import kv_oracle as O
        O.build()
        torch.set_num_threads(os.cpu_count() or 1)      # not the launcher's OMP_NUM_THREADS (torchrun exports 1)
        self.threads = torch.get_num_threads()
        self.O, self.torch = O, torch
        torch.manual_seed(0)
        self.net = ChessNet().eval()
        cfg = O.mcts_cfg(sims, temp_plies=30, max_plies=MAX_PLIES, seed=seed)
        self.sims, self.n_games = sims, n_games
        if start_lines is None:
            # the device window starts after `warm-up` self-play moves; here: after 5 uniformly random legal plies
            # (oracle-driven, seed 1234), so that the games do not share their first searches either
            start_lines = random_start_lines(n_games, 5, 1234)
            self.start = "each game after 5 uniformly random legal plies from the initial position (seed 1234)"
        else:
            self.start = "the positions of the first games at the start of the device arm's timed region"
        self.trees = [O.Tree(cfg, start_lines[g % len(start_lines)], g) for g in range(n_games)]
        self.cache = {}
        self.evals = self.served = 0
        self._sims0 = 0

    def total_sims(self):
        return sum(t_["ply"] * self.sims + t_["sims_done"] for t_ in (t.info() for t in self.trees))

    def wave(self):
        """One simulation (at least) for every live game; returns the number of leaves that went to the network."""
        from knightvision_b200.model import fp32_reference_forward
        O, torch = self.O, self.torch
        pend = []
        for t in self.trees:
            r = t.select()
            if r is None:               # the move's simulations are done: play it, start the next search
                if not t.finish_move():
                    continue
                r = t.select()
            if r is False or r is None:
                continue
            line, idx = r
            pend.append((t, line.copy(), idx.copy()))
        miss, keys = {}, []
        for t, line, idx in pend:
            k = line[:12].tobytes()
            keys.append(k)
            if k not in self.cache and k not in miss:
                miss[k] = line
        if miss:
            lines = np.stack(list(miss.values()))
            with torch.no_grad():
                pol, val = fp32_reference_forward(self.net, torch.from_numpy(O.encode(lines)))
            pol, val = pol.numpy(), val.numpy().reshape(-1)
            for j, k in enumerate(miss):
                self.cache[k] = (pol[j].copy(), float(val[j]))
        self.evals += len(miss)
        self.served += len(pend) - len(miss)
        for (t, line, idx), k in zip(pend, keys):
            lg, v = self.cache[k]
            t.expand(lg[idx], v)
        return len(miss)

    def run_waves(self, n):
        s0, e0 = self.total_sims(), self.evals
        t0 = time.perf_counter()
        for _ in range(n):
            self.wave()
        dt = time.perf_counter() - t0
        return self.total_sims() - s0, self.evals - e0, dt


def cpu_baseline(sims, budget_s=15.0, start_lines=None):
    """~budget_s of the CPU arm (see CpuSelfPlay), after one untimed wave."""
    arm = CpuSelfPlay(sims, start_lines=start_lines)
    arm.run_waves(1)
    done_s = done_e = waves = 0
    t = 0.0
    while t < budget_s:
        s_, e_, dt = arm.run_waves(2)
        done_s += s_; done_e += e_; t += dt; waves += 2
    return {"value": done_s / t, "unit": "sims/s", "cores": arm.threads, "kind": "port",
            "sample": (f"{arm.n_games} games ({arm.start}) x {waves} search waves of an {sims}-sim PUCT search "
                       f"({done_s} simulations, {done_e} network evaluations, {t:.1f} s): sequential oracle "
                       f"(oracle/kv_oracle.c) + the reference net graph in fp32 on torch CPU kernels, {arm.threads} threads, "
                       "leaves of a wave batched, positions evaluated once"),
            "net_evals_per_s": done_e / t, "evals_per_sim": done_e / done_s if done_s else None,
            "value_per_core": done_s / t / max(arm.threads, 1)}


def run_reference(args):
    """bench.py --impl reference: the CPU arm above; one step = a fixed number of search waves sized (during the warm-up)
    to about 4 s, so that the driver's --steps 20 --warmup 5 run ends within a few minutes."""
    arm = CpuSelfPlay(SIMS)
    arm.run_waves(1)
    _, _, dt = arm.run_waves(2)
    per_step = max(2, int(round(4.0 / max(dt / 2, 1e-3))))
    for _ in range(max(0, args.warmup - 1)):
        arm.run_waves(per_step)
    tot_s = tot_e = 0
    tot_t = 0.0
    for _ in range(max(1, args.steps)):
        s_, e_, dt = arm.run_waves(per_step)
        tot_s += s_; tot_e += e_; tot_t += dt
    value = tot_s / tot_t
    steps = max(1, args.steps)
    base = {"value": value, "unit": "sims/s", "cores": arm.threads, "kind": "port",
            "sample": (f"{arm.n_games} games ({arm.start}), {per_step} search waves per step of an {SIMS}-sim PUCT "
                       f"search ({tot_s} simulations, {tot_e} network evaluations in {tot_t:.1f} s): sequential oracle "
                       f"(oracle/kv_oracle.c) + the reference net graph in fp32 on torch CPU kernels, {arm.threads} threads, "
                       "leaves of a wave batched, positions evaluated once"),
            "net_evals_per_s": tot_e / tot_t, "evals_per_sim": tot_e / tot_s if tot_s else None,
            "value_per_core": value / max(arm.threads, 1),
            "note": "uses every host core of the box it runs on: boxes with more GPUs have more cores, so compare per core"}
    line = {"impl": "reference", "metric": "mcts_sims_per_s", "value": value, "unit": "sims/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * tot_t / steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"self-play, {SIMS} PUCT sims/move, reference net (random init seed 0); {arm.start}",
                       "sims_per_move": SIMS, "games": arm.n_games, "waves_per_step": per_step},
            "cpu_baseline": base,
            "e2e": {"value": value, "unit": "sims/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


DUMP_RECORDS = 8192     # records --dump-outputs writes at most: their planes are 25 MB


def dump_games(n_games, moves):
    """Games --dump-outputs writes after `moves` moves since the reset: all of them, or a fixed sample (seed 0) of
    DUMP_RECORDS // moves games, ascending.  A game records at most one position per move, so the sample holds at most
    DUMP_RECORDS records; it depends on the bench's arguments only, not on how the games went."""
    k = max(1, min(n_games, DUMP_RECORDS // max(moves, 1)))
    if k == n_games:
        return np.arange(n_games)
    return np.sort(np.random.default_rng(0).choice(n_games, k, replace=False))


def collect_outputs(eng, moves):
    """bench.py --dump-outputs: host copies of what a caller of the self-play path holds after the last move, for the
    games of dump_games (this rank's games: with several GPUs, rank 0's shard).
      games          float64 [S]          the sampled games (index within this rank's games)
      roots          float32 [S, 64]      their current positions: the 16 int64 words as 16-bit limbs (exact)
      counters       float64 [6]          over all games: done, plies played, edge-pool overflows, white wins, black
                                          wins, draws
      record_planes  float32 [R, 12, 8, 8] \\
      record_move    float64 [R]            every record of the sampled games in the reference's format (planes, move
      record_reward  float32 [R]            index, reward; SelfPlay.records), in game order, and the game it belongs to
      record_game    float64 [R]          /
    Under 28 MB in all (at most DUMP_RECORDS records)."""
    import torch
    games = dump_games(eng.mcts_games, moves)
    lines, move, reward, game = eng.mcts_records()
    sel = torch.nonzero(torch.isin(game, torch.from_numpy(games).to(game.device, game.dtype)))[:, 0]
    st = eng.mcts_status()
    return {
        "games": games.astype(np.float64),
        "roots": eng.mcts_roots().cpu().numpy()[games].view(np.uint16).astype(np.float32),
        "counters": np.array([st[k] for k in ("done", "plies", "overflow", "white_wins", "black_wins", "draws")],
                             np.float64),
        "record_planes": eng.encode(lines[sel].contiguous()).cpu().numpy(),
        "record_move": move[sel].cpu().numpy().astype(np.float64),
        "record_reward": reward[sel].cpu().numpy(),
        "record_game": game[sel].cpu().numpy().astype(np.float64),
    }


def save_outputs(out_dir, outputs):
    """collect_outputs' arrays as out_dir/<name>.npy."""
    for name, a in outputs.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def _gather_list(x, world, dev):
    """all_gather of one float per rank -> python list (rank order)."""
    import torch
    import torch.distributed as dist
    t = torch.tensor([float(x)], dtype=torch.float64, device=dev)
    if world == 1:
        return [float(x)]
    out = [torch.zeros_like(t) for _ in range(world)]
    dist.all_gather(out, t)
    return [float(o.item()) for o in out]


def run(args, rank, world, local_rank):
    import torch
    import torch.distributed as dist
    from bench import Clocks, measured_peaks
    from knightvision_b200 import parallel as P
    from knightvision_b200.engine import Engine
    from knightvision_b200.model import ChessNet
    from knightvision_b200.selfplay import SelfPlay

    G = GAMES_PER_GPU
    eng = Engine(local_rank)
    dev = eng.device
    torch.manual_seed(0)
    net = ChessNet().eval()
    sp = SelfPlay(net, G, dev, sims=SIMS, max_plies=MAX_PLIES, seed=42, engine=eng)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def distribute_weights():
        """Generation start (BASELINE config 4): the trainer rank folds its fp32 parameters once (BatchNorm folded, tower
        to bf16) and the FOLDED blob (52 MB, half the fp32 state_dict) goes to every other rank's weight arena over NCCL;
        the receivers adopt it without folding.  Returns (commit_ms, broadcast_ms) measured on this rank."""
        t0 = time.perf_counter()
        if rank == 0:
            net.mark_weights_changed()
            net.sync_weights()                       # host fp32 parameters -> device staging blob -> fold kernels
        torch.cuda.synchronize()
        commit = (time.perf_counter() - t0) * 1e3
        bcast = 0.0
        if world > 1:
            dist.barrier()                           # the other ranks wait for the fold here, not inside the broadcast timing
            torch.cuda.synchronize()
            t1 = time.perf_counter()
            dist.broadcast(eng.net_folded_tensor(), src=0)
            if rank != 0:
                eng.net_adopt_folded()
            torch.cuda.synchronize()
            bcast = (time.perf_counter() - t1) * 1e3
        return commit, bcast

    def timed_moves(n_moves, profile=False):
        """n_moves moves for every game; returns (device ms, status before, status after, per-kernel profile, launches)."""
        s0 = eng.mcts_status()
        if profile:
            eng.profile(True)
            eng.profile_read()
        l0 = eng.launches
        barrier()
        a_, b_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a_.record()
        for _ in range(n_moves):
            eng.mcts_run_move()
        b_.record()
        barrier()
        prof_ = eng.profile_read() if profile else None
        if profile:
            eng.profile(False)
        return a_.elapsed_time(b_), s0, eng.mcts_status(), prof_, eng.launches - l0

    distribute_weights()
    warm = max(args.warmup, 3)
    clocks = Clocks(local_rank)
    # ---- A: BASELINE config 3 — all games from the initial position, evaluation cache on ------------------------
    eng.mcts_enable_cache(CACHE_LOG2)
    eng.mcts_reset(None, game_id_base=rank * G)
    for _ in range(warm):
        eng.mcts_run_move()
    torch.cuda.synchronize()
    # first use of the record kernels and of the NCCL point-to-point channels behind gather (connection set-up is seconds)
    P.gather_records(*eng.mcts_records()[:3], rank * G, eng.mcts_records()[3], dst=0)
    snapshot_h = eng.mcts_roots().cpu().pin_memory()      # positions at the start of the timed region (for B and C)
    clocks.start()
    dev_ms, st0, st1, prof, launches = timed_moves(args.steps, profile=True)
    # host copies now (phase B resets the games); the files are written once the clock sampler has stopped
    outputs = collect_outputs(eng, warm + args.steps) if args.dump_outputs and rank == 0 else None
    # simulations actually run, from the device's ply counter: a game plays a ply only after its SIMS simulations, and a
    # game that ended inside the window stops contributing
    positions = st1["plies"] - st0["plies"]
    sims_done = positions * SIMS
    evals = st1["evals"] - st0["evals"]
    hits = st1["cache_hits"] - st0["cache_hits"]

    # ---- A2 (opt-in, KV_BENCH_COMPARE=1): the same moves with the pipelined schedule ----------------------------------
    alt = None
    if os.getenv("KV_BENCH_COMPARE", "0") != "0" and G >= 2048:
        eng.mcts_set_pipeline(1)
        eng.mcts_cache_clear()
        eng.mcts_reset(None, game_id_base=rank * G)
        for _ in range(warm):
            eng.mcts_run_move()
        s_ms, s0_, s1_, _, _ = timed_moves(args.steps)
        alt = {"ms_per_step": s_ms / args.steps, "sims": (s1_["plies"] - s0_["plies"]) * SIMS,
               "evals": s1_["evals"] - s0_["evals"]}
        eng.mcts_set_pipeline(-1)

    # ---- B: e2e = one generation of BASELINE config 4 through the public API with HOST buffers, everything inside the
    # timed region: weights (host fp32 parameters -> fold on the trainer rank -> NCCL broadcast of the folded blob ->
    # adopt), pinned host start positions -> device, cold evaluation cache, the same number of moves, every rank's packed
    # records gathered on rank 0 over NCCL, expanded to the reference's (planes, move, reward) tuples on the host.
    e2e_steps = args.steps
    barrier()
    t0 = time.perf_counter()
    commit_ms, bcast_ms = distribute_weights()      # clears the evaluation cache as well (new weights)
    d = snapshot_h.to(dev, non_blocking=True)
    eng.mcts_reset(d, game_id_base=rank * G)
    e0 = eng.mcts_status()
    for _ in range(e2e_steps):
        eng.mcts_run_move()
    e1 = eng.mcts_status()
    torch.cuda.synchronize()
    tg = time.perf_counter()
    lines_r, move_r, reward_r, game_r = eng.mcts_records()
    torch.cuda.synchronize()
    records_ms = (time.perf_counter() - tg) * 1e3
    if world > 1:
        dist.barrier()                               # ranks finish their moves at different times: not part of the gather
    tg = time.perf_counter()
    got = P.gather_records(lines_r, move_r, reward_r, rank * G, game_r, dst=0)
    torch.cuda.synchronize()
    gather_ms = (time.perf_counter() - tg) * 1e3
    tt = time.perf_counter()
    rec, d2h = 0, 0
    if rank == 0:
        from knightvision_b200.selfplay import records_to_tuples
        gl, gm, gr, gg = got
        recs = records_to_tuples(eng, gl, gm, gr)                   # D2H: the reference's float planes + move + reward
        rec = len(recs)
        d2h = rec * (12 * 64 * 4 + 4 + 4)
        del recs
    torch.cuda.synchronize()
    tuples_ms = (time.perf_counter() - tt) * 1e3
    e2e_s = time.perf_counter() - t0
    clk = clocks.stop()
    if outputs is not None:
        save_outputs(args.dump_outputs, outputs)
    e2e_positions = e1["plies"] - e0["plies"]
    gather_bytes = int(lines_r.shape[0]) * (16 * 8 + 4 + 4 + 8)

    # ---- C: the same positions with the evaluation cache OFF (one network evaluation per simulation) -----------------
    nocache = None
    if CACHE_LOG2:
        eng.mcts_enable_cache(0)
        eng.mcts_reset(snapshot_h.to(dev), game_id_base=rank * G)
        eng.mcts_run_move()
        n_ms, n0, n1, _, _ = timed_moves(1)
        nocache = {"ms": n_ms, "sims": (n1["plies"] - n0["plies"]) * SIMS, "evals": n1["evals"] - n0["evals"]}

    # ---- D: "random positions" variant (SURVEY §8d): k in [0,40) random legal plies per game, seed 1234, cache on ----
    eng.mcts_enable_cache(CACHE_LOG2)
    eng.mcts_reset(eng.random_positions(G, 40, 1234 + rank), game_id_base=rank * G)
    for _ in range(warm):
        eng.mcts_run_move()
    r_moves = max(1, min(args.steps, 2))
    r_ms, r0, r1, _, _ = timed_moves(r_moves)
    r_sims = (r1["plies"] - r0["plies"]) * SIMS
    r_evals = r1["evals"] - r0["evals"]

    # ---- E: few games, K simulations in flight per game with virtual loss (G/K games x K = the same leaves per wave) ----
    K = INFLIGHT
    vl = None
    if K > 1 and G % K == 0:
        Gk = G // K
        eng.mcts_create(Gk, SIMS, MAX_PLIES, seed=42, eval_mode=1, inflight=K)
        eng.mcts_enable_cache(CACHE_LOG2)
        eng.mcts_reset(None, game_id_base=rank * Gk)
        for _ in range(warm):
            eng.mcts_run_move()
        w0 = eng.mcts_waves()
        v_moves = max(1, min(args.steps, 3))
        v_ms, v0, v1, _, _ = timed_moves(v_moves)
        vl = {"games_per_gpu": Gk, "inflight": K, "ms_per_step": v_ms / v_moves, "moves": v_moves,
              "sims": (v1["plies"] - v0["plies"]) * SIMS, "evals": v1["evals"] - v0["evals"],
              "waves_per_move": (eng.mcts_waves() - w0) / v_moves}

    # ---- F: the reference's own move rule (scripts/self_play.py:147-189): no search, one network evaluation per ply,
    # root priors mixed over all 4096 indices as the reference does, resignation on (sims = 1).  positions/s here is
    # directly comparable with the reference's self-play loop (BASELINE configs[0]).
    pm = None
    if POLICY_MODE_PLIES > 0:
        eng.mcts_create(G, 1, MAX_PLIES, seed=42, eval_mode=1)
        eng.mcts_enable_cache(0)
        eng.mcts_reset(None, game_id_base=rank * G)
        for _ in range(warm):
            eng.mcts_run_move()
        p_ms, p0, p1, _, _ = timed_moves(POLICY_MODE_PLIES)
        pm = {"ms": p_ms, "positions": p1["plies"] - p0["plies"], "evals": p1["evals"] - p0["evals"]}

    t = torch.tensor([dev_ms, e2e_s * 1e3, nocache["ms"] if nocache else 0.0, r_ms, commit_ms, bcast_ms, gather_ms,
                      records_ms, tuples_ms], dtype=torch.float64, device=dev)
    cnt = torch.tensor([float(sims_done), float(evals), float(positions), float(rec), float(hits), float(r_sims),
                        float(r_evals), float(e2e_positions), float(st1["overflow"]), float(st0["done"]), float(st1["done"]),
                        float(gather_bytes), float(nocache["sims"] if nocache else 0)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(cnt, op=dist.ReduceOp.SUM)
    per_rank_ms = _gather_list(dev_ms / args.steps, world, dev)
    per_rank_mhz = _gather_list(clk.get("sm_mhz") or 0.0, world, dev)
    per_rank_conv = _gather_list(prof["net_conv"][0] / args.steps, world, dev)
    dev_ms, e2e_ms, nocache_ms, r_ms, commit_ms, bcast_ms, gather_ms, records_ms, tuples_ms = (float(x) for x in t)
    (sims_all, evals_all, pos_all, rec_all, hits_all, r_sims_all, r_evals_all, e2e_pos_all, overflow_all, done0_all,
     done1_all, gather_bytes_all, nocache_sims_all) = (float(x) for x in cnt)
    sub = sub_records(args, eng, rank, world, local_rank) if os.getenv("KV_BENCH_SUB", "1") != "0" else None
    if rank != 0:
        return
    peaks = measured_peaks()
    conv_ms, conv_n = prof["net_conv"]
    traffic, traffic_src = _ncu_traffic()
    achieved = (evals * CONV_FLOPS_PER_EVAL) / (conv_ms * 1e-3) / 1e12 if conv_ms > 0 else 0.0
    value = sims_all / (dev_ms * 1e-3)
    ceiling_evals = achieved * 1e12 / CONV_FLOPS_PER_EVAL if achieved else None     # evals/s at the tower kernel's own rate
    line = {
        "metric": "mcts_sims_per_s", "value": value, "unit": "sims/s", "n_gpus": world, "steps": args.steps,
        "warmup": warm, "ms_per_step": dev_ms / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": {"workload": (f"self-play: {G} concurrent games per GPU, {SIMS} PUCT sims/move, reference ChessNet "
                                "(random init seed 0, BN folded, bf16 tower / fp32 accumulate), all games from the initial "
                                f"position; one step = one move for every game; timed window = moves {warm + 1}..{warm + args.steps}"),
                   "games_per_gpu": G, "sims_per_move": SIMS, "parallelism": f"games sharded by id over {world} GPU(s)",
                   "l2": "working set (node/edge pools + activations, > 3 GB) exceeds the 126 MB L2; no flush needed"},
        "sims_counted": "device ply counter x sims per move (a ply is played only after its simulations ran)",
        "games": {"per_gpu": G, "done_before": done0_all, "done_after": done1_all, "overflow": overflow_all,
                  "note": "done = games that ended (mate / stalemate / only kings / resignation / ply cap) before / after the "
                          "timed window, summed over ranks; overflow = games whose edge pool overflowed (search truncated)"},
        "positions_per_s": pos_all / (dev_ms * 1e-3), "net_evals_per_s": evals_all / (dev_ms * 1e-3),
        "evals_per_sim": evals_all / sims_all if sims_all else None,
        "per_rank": {"ms_per_step": per_rank_ms, "sm_mhz_median": per_rank_mhz, "tower_kernel_ms_per_step": per_rank_conv,
                     "note": "value uses the slowest rank (max over ranks); no collective runs inside the timed window"},
        "ceiling": ({"net_evals_per_s_at_kernel_rate": ceiling_evals,
                     "sims_per_s_at_this_evals_per_sim": ceiling_evals / (evals_all / sims_all) if evals_all else None,
                     "achieved_fraction": (value / world) / (ceiling_evals / (evals_all / sims_all)) if evals_all else None,
                     "evals_per_sim_needed_for_1e6_sims_per_s": ceiling_evals / 1e6,
                     "note": "per GPU: the tensor-core tower bounds evaluations/s; sims/s = evaluations/s / (evaluations per "
                             "simulation).  1e6 sims/s/GPU needs the evaluation cache to serve all but this share of the "
                             "simulations"} if ceiling_evals else None),
        "eval_cache": {"log2_slots": CACHE_LOG2, "bytes": (640 << CACHE_LOG2) if CACHE_LOG2 else 0,
                       "served_per_sim": hits_all / sims_all if sims_all else None,
                       "note": "keyed by the 12 bitboards (the net's whole input); search results are bit-identical "
                               "with the cache on or off (tests/test_gpu_mcts.py::test_eval_cache_is_transparent)"},
        "schedule": {"tower": ("one dependency-scheduled launch per evaluation batch (tower_umma2_kernel<halo>: depth-first "
                               "chunks, activation tiles fetched 3x instead of 9x per channel block)"),
                     "pipelined": False,
                     "pipelined_alt": ({"value": world * alt["sims"] / (alt["ms_per_step"] * args.steps * 1e-3),
                                        "unit": "sims/s", "ms_per_step": alt["ms_per_step"],
                                        "evals_per_sim": alt["evals"] / alt["sims"] if alt["sims"] else None,
                                        "note": "rank 0's figures x world, kv_mcts_set_pipeline(1)"} if alt else None)},
        "no_cache": ({"value": nocache_sims_all / (nocache_ms * 1e-3), "unit": "sims/s", "ms_per_step": nocache_ms,
                      "evals_per_sim": nocache["evals"] / nocache["sims"] if nocache["sims"] else None,
                      "note": "same positions, evaluation cache disabled"} if nocache else None),
        "random_positions": {"value": r_sims_all / (r_ms * 1e-3), "unit": "sims/s",
                             "evals_per_sim": r_evals_all / r_sims_all if r_sims_all else None,
                             "ms_per_step": r_ms / r_moves,
                             "note": "every game starts after k in [0,40) uniformly random legal plies (seed 1234), "
                                     "cache on, same warm-up"},
        "virtual_loss": ({"value": world * vl["sims"] / (vl["ms_per_step"] * 1e-3 * vl["moves"]), "unit": "sims/s",
                          "games_per_gpu": vl["games_per_gpu"], "inflight": vl["inflight"],
                          "ms_per_step": vl["ms_per_step"], "evals_per_sim": vl["evals"] / vl["sims"] if vl["sims"] else None,
                          "waves_per_move": vl["waves_per_move"],
                          "note": "rank 0's figures x world: G/K games with K simulations in flight per game and wave "
                                  "(virtual loss), initial position, cache on"} if vl else None),
        "policy_mode": ({"value": world * pm["positions"] / (pm["ms"] * 1e-3), "unit": "positions/s", "plies": POLICY_MODE_PLIES,
                         "evals_per_position": pm["evals"] / pm["positions"] if pm["positions"] else None,
                         "note": "rank 0's figures x world: sims = 1, the reference's own rule (scripts/self_play.py:147-189: no "
                                 "search, one network evaluation per ply, softmax and Dirichlet noise over all 4096 indices, legal "
                                 "renormalisation, sampling, resignation below -0.7 after move 15); SURVEY section 6 measured 48.6 "
                                 "positions/s for the unmodified reference on 8 CPU threads"} if pm else None),
        "clocks": clk, "gpu_launches": launches,
        "e2e": {"value": e2e_pos_all * SIMS / (e2e_ms * 1e-3), "unit": "sims/s",
                "h2d_bytes_per_step": (G * 128 + (int(eng._lib.kv_net_blob_floats(eng.ctx)) * 4)) // e2e_steps,
                "d2h_bytes_per_step": d2h // e2e_steps, "records_returned": rec_all, "steps": e2e_steps,
                "commit_ms": commit_ms, "broadcast_ms": bcast_ms,
                "broadcast_bytes": int(eng._lib.kv_net_folded_bytes(eng.ctx)) if world > 1 else 0,
                "records_ms": records_ms, "gather_ms": gather_ms, "gather_bytes": gather_bytes_all, "tuples_ms": tuples_ms,
                "phases_note": ("commit = fp32 parameters (host) -> device -> fold, on the trainer rank; broadcast = NCCL broadcast "
                                "of the folded blob + adopt; records = per-rank compaction of the game records on the device; "
                                "gather = NCCL gather of the packed records to rank 0; tuples = kv_encode + D2H + building the "
                                "reference's tuple list on rank 0 (max over ranks each)"),
                "api": ("one generation through the public API with host buffers: fp32 parameters (host) -> fold on the trainer "
                        "rank -> NCCL broadcast of the folded bf16 blob -> adopt; pinned host start lines -> kv_mcts_reset -> "
                        "steps x kv_mcts_run_move (cold evaluation cache) -> packed records gathered on rank 0 over NCCL "
                        "(parallel.gather_records) -> kv_encode -> the reference's (planes, move, reward) tuples on the host; "
                        "max over ranks of the wall time")},
        "roofline": {"kernel": ("tower_umma2_kernel (tcgen05 cta_group::2 implicit GEMM, the 11 tower convolutions of one "
                                "evaluation batch in one dependency-scheduled launch)"), "bound": "tensor", "achieved": achieved,
                     "peak": peaks["bf16_sustained"], "unit": "TFLOP/s", "frac": achieved / peaks["bf16_sustained"],
                     "traffic": traffic, "traffic_source": (f"{traffic_src}: dram__bytes_read.sum + dram__bytes_write.sum of one "
                                                             f"launch over {G} boards (a wave of the search "
                                                             "evaluates fewer: evals_per_sim x games).  If every layer went through "
                                                             "HBM the launch would move 7.1 GB (2.8 in + 2.95 out + 1.34 residual + "
                                                             "0.05 weights); depth-first chunks keep a chunk's activations in L2")
                     if traffic else None,
                     "peak_source": peaks["source"] + ", sustained bf16 figure",
                     "kernel_ms_per_step": conv_ms / args.steps, "kernel_share_of_step": conv_ms / dev_ms,
                     "flops_per_eval_in_kernel": CONV_FLOPS_PER_EVAL, "launches": conv_n},
        "kernels_ms_per_step": {k: v[0] / args.steps for k, v in prof.items() if v[1]},
        "cpu_baseline": cpu_baseline(SIMS, start_lines=snapshot_h.numpy().view(np.uint64)[:CPU_GAMES].copy()) if world == 1 else None,
        "sub": sub,
    }
    print(json.dumps(line), flush=True)


def sub_records(args, eng, rank, world, local_rank):
    """BASELINE configs[1] (perft) and configs[4] (training step, learn loop) as short sub-records of the default run, so the
    driver-run line carries them at every N.  Each has its own roofline / e2e (and cpu_baseline at N = 1)."""
    import bench
    import bench_learn
    import bench_train
    out = {}
    steps = max(2, min(args.steps, 5))
    for name, fn in (("perft", lambda: bench.perft_record(args, eng, rank, world, steps=steps, cpu=(world == 1))),
                     ("movegen", lambda: bench.rules_record(args, eng, rank, world, steps=steps)),
                     ("train", lambda: bench_train.train_record(args, eng, rank, world, local_rank, steps=6, arms=("native",),
                                                                graph=False)),
                     ("learn", lambda: bench_learn.learn_record(args, eng, rank, world, local_rank, warm=1, steps=1, plies=1))):
        if os.getenv("KV_BENCH_SUB_" + name.upper(), "1") == "0":
            continue
        try:
            out[name] = fn()
        except Exception as e:              # a failing sub-phase must not lose the headline line; it is reported, not hidden
            import traceback
            out[name] = {"error": f"{type(e).__name__}: {e}"[:300], "trace": traceback.format_exc()[-600:]}
    return out
