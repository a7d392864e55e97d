"""ctypes wrapper of the CPU parity oracle (oracle/kv_oracle.c).

TEST INFRASTRUCTURE ONLY: importable from tests/, __graft_entry__.smoke() and bench.py's CPU legs.
Nothing under knightvision_b200/ imports this module.
"""
from __future__ import annotations

import ctypes
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "libkv_oracle.so")


def build(force: bool = False) -> str:
    deps = [os.path.join(_HERE, "kv_oracle.c"), os.path.join(_HERE, "..", "include", "kv_detmath.h")]
    if force or not os.path.exists(_SO) or any(os.path.getmtime(_SO) < os.path.getmtime(d) for d in deps):
        subprocess.check_call(["make", "-C", _HERE, "-s", "-B", "libkv_oracle.so"])
    return _SO


_lib = None


def lib():
    global _lib
    if _lib is None:
        _lib = ctypes.CDLL(build())
        _lib.kvo_square_under_attack.restype = ctypes.c_int
        _lib.kvo_in_check.restype = ctypes.c_int
        _lib.kvo_move_index.restype = ctypes.c_int
    return _lib


def _p(a):
    return a.ctypes.data_as(ctypes.c_void_p)


MOVE_STRIDE = 256


def movegen(lines: np.ndarray):
    """lines: uint64 [n,16] (modified in place only in the documented king-resurrection corner).
    Returns (moves u16 [n,256], counts i32 [n], flags i32 [n])."""
    lines = np.ascontiguousarray(lines, dtype=np.uint64)
    n = lines.shape[0]
    moves = np.zeros((n, MOVE_STRIDE), dtype=np.uint16)
    counts = np.zeros(n, dtype=np.int32)
    flags = np.zeros(n, dtype=np.int32)
    lib().kvo_movegen(_p(lines), ctypes.c_int(n), _p(moves), ctypes.c_int(MOVE_STRIDE), _p(counts), _p(flags))
    return moves, counts, flags, lines


def make_moves(lines: np.ndarray, mv: np.ndarray) -> np.ndarray:
    out = np.ascontiguousarray(lines, dtype=np.uint64).copy()
    mv = np.ascontiguousarray(mv, dtype=np.uint16)
    lib().kvo_make_moves(_p(out), ctypes.c_int(out.shape[0]), _p(mv))
    return out


def perft(line: np.ndarray, depth: int) -> np.ndarray:
    """Returns uint64[6]: nodes, captures, ep, castles, promos, order digest."""
    line = np.ascontiguousarray(line, dtype=np.uint64)
    out = np.zeros(6, dtype=np.uint64)
    lib().kvo_perft(_p(line), ctypes.c_int(depth), _p(out))
    return out


def perft2(line: np.ndarray, depth: int) -> np.ndarray:
    """Returns uint64[8] in the layout of kv_perft (include/kv_b200.h)."""
    line = np.ascontiguousarray(line, dtype=np.uint64)
    out = np.zeros(8, dtype=np.uint64)
    lib().kvo_perft2(_p(line), ctypes.c_int(depth), _p(out))
    return out


def square_under_attack(line: np.ndarray, r: int, c: int) -> bool:
    line = np.ascontiguousarray(line, dtype=np.uint64)
    return bool(lib().kvo_square_under_attack(_p(line), ctypes.c_int(r), ctypes.c_int(c)))


def in_check(line: np.ndarray) -> bool:
    line = np.ascontiguousarray(line, dtype=np.uint64)
    return bool(lib().kvo_in_check(_p(line)))


def encode(lines: np.ndarray) -> np.ndarray:
    lines = np.ascontiguousarray(lines, dtype=np.uint64)
    n = lines.shape[0]
    out = np.zeros((n, 12, 8, 8), dtype=np.float32)
    lib().kvo_encode(_p(lines), ctypes.c_int(n), _p(out))
    return out


# ---- MCTS oracle (oracle/kv_oracle.c, "parity unpinned": the specification of the new tree search) -----------
class MctsCfg(ctypes.Structure):
    _fields_ = [("sims", ctypes.c_int32), ("edge_cap", ctypes.c_int32), ("temp_plies", ctypes.c_int32),
                ("max_plies", ctypes.c_int32), ("c_puct", ctypes.c_float), ("dir_alpha", ctypes.c_float),
                ("dir_eps", ctypes.c_float), ("inflight", ctypes.c_int32), ("seed", ctypes.c_uint64),
                ("resign_thr", ctypes.c_float), ("resign_min_plies", ctypes.c_int32), ("root_mix", ctypes.c_int32),
                ("pad", ctypes.c_int32)]


def mcts_cfg(sims, edges_per_node=64, temp_plies=0, max_plies=1 << 20, c_puct=1.5, dir_alpha=0.3, dir_eps=0.25, seed=1,
             inflight=1, resign_thr=-0.7, resign_min_plies=15, root_mix=-1):
    """Defaults follow kv_mcts_create_k: the reference's resign rule (scripts/self_play.py:184-189) and, when sims == 1,
    its prior mixing over all 4096 indices (:150-167)."""
    return MctsCfg(sims, max(sims * (edges_per_node or 64), 256), temp_plies, max_plies, c_puct, dir_alpha, dir_eps,
                   inflight, seed, resign_thr, resign_min_plies, int(sims == 1) if root_mix < 0 else root_mix, 0)


def mcts_search(cfg, line, game_id=0, ply=0, replay=None, nodes=False):
    """One search.  replay = (node_val f32[], node_first i32[], edge_P f32[]) dumps of the device tree, or None for
    the hash evaluator.  Returns dict(move, moves, N, W, P, nodes, edges, overflow).
    nodes=True adds the whole tree, numbered in creation order as on the device: node_line u64 [nodes,16] (the line as
    stored after move generation, i.e. the position the evaluator sees), node_term, node_first (-1 none), node_n
    (edge count), node_N, node_val (terminal or evaluator value, side to move's view); edge_mv, edge_child (-1
    unexpanded), edge_P, edge_W, edge_N [edges]."""
    line = np.ascontiguousarray(line, dtype=np.uint64)
    moves = np.zeros(256, np.uint16); N = np.zeros(256, np.uint32); W = np.zeros(256, np.float32)
    P = np.zeros(256, np.float32); info = np.zeros(4, np.int32)
    if replay is None:
        rv = rf = rp = None
    else:
        rv, rf, rp = (np.ascontiguousarray(replay[0], np.float32), np.ascontiguousarray(replay[1], np.int32),
                      np.ascontiguousarray(replay[2], np.float32))
    args = [ctypes.byref(cfg), _p(line), ctypes.c_uint64(game_id), ctypes.c_int(ply),
            _p(rv) if rv is not None else None, _p(rf) if rf is not None else None, _p(rp) if rp is not None else None,
            _p(moves), _p(N), _p(W), _p(P), _p(info)]
    if nodes:
        nc, ec = int(cfg.sims) + 1, int(cfg.edge_cap)
        t = dict(node_line=np.zeros((nc, 16), np.uint64), node_i32=np.zeros((nc, 4), np.int32),
                 node_val=np.zeros(nc, np.float32), edge_mv=np.zeros(ec, np.uint16), edge_child=np.zeros(ec, np.int32),
                 edge_P=np.zeros(ec, np.float32), edge_W=np.zeros(ec, np.float32), edge_N=np.zeros(ec, np.uint32))
        f = lib().kvo_mcts_search_tree
        args += [_p(a) for a in t.values()]
    else:
        f = lib().kvo_mcts_search
    f.restype = ctypes.c_int
    mv = f(*args)
    n = int(info[0])
    out = dict(move=mv, moves=moves[:n], N=N[:n], W=W[:n], P=P[:n], nodes=int(info[1]), edges=int(info[2]),
               overflow=int(info[3]))
    if nodes:
        nn, ne = out["nodes"], out["edges"]
        ni = t.pop("node_i32")[:nn]
        out.update(node_term=ni[:, 0].astype(bool), node_first=ni[:, 1], node_n=ni[:, 2], node_N=ni[:, 3].astype(np.uint32))
        out.update({k: v[:nn] if k.startswith("node") else v[:ne] for k, v in t.items()})
    return out


def root_eta(alpha, seed, game_id, ply, n):
    """Root noise eta[k] (k < n legal moves) of the legal-move prior rule: Gamma(alpha) variates keyed by ply * 256 + k,
    divided by their sequential float32 sum.  Root priors are (1 - eps) * softmax + eps * eta."""
    out = np.zeros(max(int(n), 1), np.float32)
    lib().kvo_root_eta(ctypes.c_float(alpha), ctypes.c_uint64(seed), ctypes.c_uint64(game_id), ctypes.c_int(ply),
                       ctypes.c_int(int(n)), _p(out))
    return out[:int(n)]


def selfplay_game(cfg, start_line, game_id=0, script_moves=None, script_vals=None, return_flags=False):
    """One game of the oracle's game loop.  script_moves (u16 words, 0xFFFF = none) / script_vals (f32, NaN = none):
    per ply the move to play instead of the search's choice and the value the resign rule sees."""
    start_line = np.ascontiguousarray(start_line, dtype=np.uint64)
    mp = int(cfg.max_plies)
    moves = np.zeros(mp, np.uint16)
    lines = np.zeros((mp, 16), np.uint64)
    res = ctypes.c_int32(0)
    flags = ctypes.c_int32(0)
    sm = np.ascontiguousarray(script_moves, np.uint16) if script_moves is not None else None
    sv = np.ascontiguousarray(script_vals, np.float32) if script_vals is not None else None
    sn = len(sm) if sm is not None else (len(sv) if sv is not None else 0)
    f = lib().kvo_selfplay_game2
    f.restype = ctypes.c_int
    n = f(ctypes.byref(cfg), _p(start_line), ctypes.c_uint64(game_id), _p(sm) if sm is not None else None,
          _p(sv) if sv is not None else None, ctypes.c_int(sn), _p(moves), _p(lines), ctypes.byref(res), ctypes.byref(flags))
    if return_flags:
        return moves[:n], lines[:n], int(res.value), int(flags.value)
    return moves[:n], lines[:n], int(res.value)


def root_noise(alpha, seed, game_id, ply):
    """Gamma(alpha) variates of the reference-rule root noise for all 4096 policy indices (key = ply * 4096 + index)."""
    src = lib().kvo_root_noise
    out = np.zeros(4096, np.float32)
    src(ctypes.c_float(alpha), ctypes.c_uint64(seed), ctypes.c_uint64(game_id), ctypes.c_int(ply), _p(out))
    return out


def hash_eval(line):
    """(logits f32[4096], white-perspective value) of the hash test evaluator for a position."""
    line = np.ascontiguousarray(line, dtype=np.uint64)
    out = np.zeros(4096, np.float32)
    f = lib().kvo_hash_eval
    f.restype = ctypes.c_float
    v = f(_p(line), _p(out))
    return out, float(v)


class Tree:
    """Step-wise sequential search with an external evaluator (kvo_tree_*): bench.py's CPU arm batches the leaves of many
    games for the fp32 network.  select() -> (line, legal policy indices) | None when the move's simulations are done."""

    def __init__(self, cfg, start_line, game_id=0):
        self.cfg = cfg
        f = lib().kvo_tree_new
        f.restype = ctypes.c_void_p
        self._line = np.ascontiguousarray(start_line, dtype=np.uint64)
        self.h = ctypes.c_void_p(f(ctypes.byref(cfg), _p(self._line), ctypes.c_uint64(game_id)))
        self._leaf = np.zeros(16, np.uint64)
        self._idx = np.zeros(256, np.int32)
        self._n = ctypes.c_int32(0)

    def close(self):
        if self.h and _lib is not None:
            _lib.kvo_tree_free(self.h)
        self.h = None

    def __del__(self):
        self.close()

    def select(self):
        """1 -> (leaf line u64[16], legal policy indices i32[n]); 0 -> None (call finish_move); game over -> False."""
        f = lib().kvo_tree_select
        f.restype = ctypes.c_int
        r = f(self.h, _p(self._leaf), _p(self._idx), ctypes.byref(self._n))
        if r == 1:
            return self._leaf, self._idx[:self._n.value]
        return None if r == 0 else False

    def expand(self, legal_logits, v_white):
        lg = np.ascontiguousarray(legal_logits, np.float32)
        lib().kvo_tree_expand(self.h, _p(lg), ctypes.c_float(v_white))

    def finish_move(self) -> bool:
        f = lib().kvo_tree_finish_move
        f.restype = ctypes.c_int
        return bool(f(self.h))

    def info(self):
        info = np.zeros(5, np.int32)
        moves = np.zeros(max(int(self.cfg.max_plies), 1), np.uint16)
        lib().kvo_tree_info(self.h, _p(info), _p(moves))
        return dict(ply=int(info[0]), done=bool(info[1]), result=int(info[2]), sims_done=int(info[3]),
                    overflow=int(info[4]), moves=moves[:int(info[0])])
