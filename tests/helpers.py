"""Shared helpers for the parity tests (oracle-driven position generators)."""
from __future__ import annotations

import json
import os

import numpy as np

from knightvision_b200 import layout as L
from oracle import kv_oracle as O

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")

PERFT_EXPECT = {"startpos": [20, 400, 8902, 197281, 4865721], "castle_w": [26, 568, 13744, 314346],
                "castle_b": [26, 568, 13744, 314346], "ep_a": [6, 38, 257, 1971], "ep_b": [6, 38, 257, 1971],
                "promo_w": [24, 462, 12448, 274548], "promo_b": [24, 462, 12448, 272623]}


def load_rows(name):
    return np.load(os.path.join(GOLDEN, name + ".npz"))


def perft_gold():
    with open(os.path.join(GOLDEN, "perft.json")) as f:
        return json.load(f)


def random_playout_positions(n_games: int, max_plies: int, seed: int) -> np.ndarray:
    """Positions visited by uniformly random playouts driven by the ORACLE (already pinned to the reference)."""
    rng = np.random.default_rng(seed)
    lines = np.stack([L.start_line()] * n_games)
    alive = np.ones(n_games, dtype=bool)
    out = []
    for _ in range(max_plies):
        if not alive.any():
            break
        cur = lines[alive]
        out.append(cur.copy())
        moves, counts, flags, mid = O.movegen(cur.copy())
        pick = np.full(len(cur), 0xFFFF, dtype=np.uint16)
        ok = counts > 0
        idx = (rng.random(len(cur)) * np.maximum(counts, 1)).astype(np.int64)
        pick[ok] = moves[np.arange(len(cur)), idx][ok]
        nxt = O.make_moves(mid, pick)
        lines[alive] = nxt
        a = alive.copy()
        a[alive] = ok & ((flags & L.RF_ONLY_KINGS) == 0)
        alive = a
    return np.concatenate(out)


def check_movegen_against(rows_or_lines, got):
    """got = (moves, counts, flags, lines_after).  Compares with the golden rows (or the oracle for raw lines)."""
    moves, counts, flags, after = got
    if isinstance(rows_or_lines, np.ndarray):
        em, ec, ef, ea = O.movegen(rows_or_lines.copy())
    else:
        r = rows_or_lines
        ec, ef, ea = r["counts"], r["flags"], r["line_mid"]
        em = np.zeros((len(ec), 256), dtype=np.uint16)
        em[:, :r["moves"].shape[1]] = r["moves"]
    assert np.array_equal(counts, ec)
    assert np.array_equal(flags, ef)
    k = np.arange(256)[None, :] < np.minimum(ec, 256)[:, None]
    assert np.array_equal(np.where(k, moves[:, :256], 0), np.where(k, em, 0))
    assert np.array_equal(after[:, :13], ea[:, :13])


def synthetic_lines(n: int, seed: int, wild: bool = True) -> np.ndarray:
    """n random board lines in the spirit of oracle/gen_golden.py:279-339 (the generator behind the reference-made
    `synthetic` fixtures), but built directly as lines: random piece placements, side, moved flags, e.p. square, and —
    when `wild` — missing kings, king *location variables* that disagree with the board, pawns on the back ranks and
    arbitrary e.p. squares.  The oracle (pinned to the reference on 3 000 such rows) is the judge for these."""
    rng = np.random.default_rng(seed)
    out = np.zeros((n, 16), dtype=np.uint64)
    kinds = np.array([1, 2, 3, 4, 5, 5, 5])          # Q R B N p p p  (index into the colour's bitboards)
    for i in range(n):
        sq = rng.permutation(64)
        bbs = [0] * 12
        wk, bk = int(sq[0]), int(sq[1])
        castle_bias = (not wild) and rng.random() < 0.5
        used = 2
        if castle_bias:
            wk, bk = 60, 4
            bbs[0] |= 1 << 60
            bbs[6] |= 1 << 4
            for s, idx in ((56, 2), (63, 2), (0, 8), (7, 8)):
                if rng.random() < 0.8:
                    bbs[idx] |= 1 << s
            free = [s for s in sq if s not in (60, 4, 56, 63, 0, 7)]
        else:
            if not (wild and rng.random() < 0.25):
                bbs[0] |= 1 << wk
            if not (wild and rng.random() < 0.25):
                bbs[6] |= 1 << bk
            free = list(sq[used:])
        for s in free[:int(rng.integers(0, 21 if wild else 15))]:
            s = int(s)
            t = int(kinds[rng.integers(0, 7)])
            if t == 5 and not wild and (s >> 3) in (0, 7):
                continue
            bbs[t + (6 if rng.random() < 0.5 else 0)] |= 1 << s
        wtm = rng.random() < 0.5
        if wild and rng.random() < 0.3:
            wk = int(rng.integers(0, 64))
        if wild and rng.random() < 0.3:
            bk = int(rng.integers(0, 64))
        moved = int(sum((1 << b) for b in range(6) if rng.random() < 0.25))
        ep = 64
        if rng.random() < 0.4:
            if wild:
                ep = int(rng.integers(0, 64))
            else:
                r, pr, c = (2, 3, int(rng.integers(0, 8))) if wtm else (5, 4, int(rng.integers(0, 8)))
                occ = 0
                for b in bbs:
                    occ |= b
                if not (occ >> (r * 8 + c)) & 1 and not (occ >> (pr * 8 + c)) & 1:
                    bbs[11 if wtm else 5] |= 1 << (pr * 8 + c)
                    ep = r * 8 + c
        clock = int(rng.choice([0, 0, 3, 99, 100, 150]))
        for k in range(12):
            out[i, k] = np.uint64(bbs[k])
        out[i, 12] = np.uint64(int(wtm) | (moved << 1) | (ep << 8) | (wk << 16) | (bk << 24) | (clock << 32))
    return out


# 218 legal moves for white (R6R/3Q4/1Q4Q1/4Q3/2Q4Q/Q4Q2/pp1Q4/kBNN1KB1 w); most replies are mates or stalemates
MANY_MOVES_BOARD = [
    ["wR", "--", "--", "--", "--", "--", "--", "wR"],
    ["--", "--", "--", "wQ", "--", "--", "--", "--"],
    ["--", "wQ", "--", "--", "--", "--", "wQ", "--"],
    ["--", "--", "--", "--", "wQ", "--", "--", "--"],
    ["--", "--", "wQ", "--", "--", "--", "--", "wQ"],
    ["wQ", "--", "--", "--", "--", "wQ", "--", "--"],
    ["bp", "bp", "--", "wQ", "--", "--", "--", "--"],
    ["bK", "wB", "wN", "wN", "--", "wK", "wB", "--"],
]


def search_roots(n_random: int = 20, seed: int = 61):
    """(lines u64 [n,16], names) of search roots where evaluators go wrong: the start position; random-playout positions,
    half with white and half with black to move; the perft golden positions (castling, e.p., promotion); a position
    with 218 legal moves; one with an e.p. capture; a synthetic line whose move generation rewrites the board (the
    getKingMoves restore quirk, RF_STATE_MUTATED: the position evaluated is not the line given); and three roots that
    share the 12 bitboards (the network's whole input and the evaluation cache's key) with another root but differ in
    side to move, castling rights or e.p. square.  (castle_w and castle_b share their bitboards too.)"""
    gold = perft_gold()
    lines, names = [L.start_line()], ["start"]
    pos = random_playout_positions(n_games=8, max_plies=90, seed=seed)
    _, counts, flags, _ = O.movegen(pos.copy())
    ok = (counts > 0) & ((flags & L.RF_ONLY_KINGS) == 0)
    rng = np.random.default_rng(seed)
    for side in (1, 0):
        cand = np.nonzero(ok & ((pos[:, 12] & np.uint64(1)) == side))[0]
        for i in rng.choice(cand, n_random // 2, replace=False):
            lines.append(pos[i])
            names.append(f"playout {i} {'white' if side else 'black'} to move")
    for k in gold:
        if k != "startpos":
            lines.append(np.array(gold[k]["line"], dtype=np.uint64))
            names.append(k)
    lines.append(L.pack_fields(MANY_MOVES_BOARD, True, wk=(7, 5), bk=(7, 0), moved=63))
    names.append("218 moves")
    ep = O.make_moves(np.array(gold["ep_a"]["line"], dtype=np.uint64)[None], np.array([L.move_word(1, 3, 3, 3)]))[0]
    lines.append(ep)                                               # white can take d7-d5 e.p. at the root
    names.append("ep_a after d7-d5")
    syn = synthetic_lines(64, 0)
    _, counts, flags, _ = O.movegen(syn.copy())
    mut = np.nonzero(((flags & L.RF_STATE_MUTATED) != 0) & (counts > 0) & ((flags & L.RF_ONLY_KINGS) == 0))[0]
    lines.append(syn[mut[0]])
    names.append(f"synthetic {mut[0]}, board rewritten by move generation")
    # same bitboards, other side to move (and no e.p. square); castling rights gone; e.p. square gone
    no_ep = ~np.uint64(0x7F00)
    flip = lines[1].copy()
    flip[12] = ((flip[12] ^ np.uint64(1)) & no_ep) | np.uint64(L.EP_NONE << 8)
    lines.append(flip)
    names.append(names[1] + ", other side to move")
    castle = np.array(gold["castle_w"]["line"], dtype=np.uint64)
    castle[12] |= np.uint64(L.F_WK << 1)
    lines.append(castle)
    names.append("castle_w, king moved")
    ep = ep.copy()
    ep[12] = (ep[12] & no_ep) | np.uint64(L.EP_NONE << 8)
    lines.append(ep)
    names.append("ep_a after d7-d5 without e.p. square")
    return np.stack(lines), names


def oracle_attack_masks(lines: np.ndarray) -> np.ndarray:
    """squareUnderAttack for all 64 squares of every line as a bit mask (bit r*8+c), from the oracle."""
    out = np.zeros(len(lines), dtype=np.uint64)
    for i, l in enumerate(lines):
        m = 0
        for s in range(64):
            if O.square_under_attack(l, s >> 3, s & 7):
                m |= 1 << s
        out[i] = np.uint64(m)
    return out
