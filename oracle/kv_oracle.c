/*
 * kv_oracle.c — CPU restatement of KnightVision's custom chess rules (TEST INFRASTRUCTURE ONLY).
 *
 * This file is the parity oracle for the B200 hot path.  It is NOT a product code path:
 * only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs
 * may load it.  The product library (libkv_b200.so) never links or calls it.
 *
 * It restates, as a plain mailbox engine in C, the algorithm of the reference
 * `core/chessEngine.py` (all file:line citations are relative to /root/reference):
 *   - state                       core/chessEngine.py:34-84
 *   - getValidMoves               core/chessEngine.py:277-321
 *   - checkForPinsAndChecks       core/chessEngine.py:325-383   (7-entry knight table, :373-374)
 *   - inCheck / squareUnderAttack core/chessEngine.py:388-415   (re-entrancy guard :401-402)
 *   - getAllPossibleMoves         core/chessEngine.py:433-441
 *   - piece generators            core/chessEngine.py:447-601
 *   - addPieceMovesConsideringPins core/chessEngine.py:604-630
 *   - makeMove                    core/chessEngine.py:127-197
 *   - checkForEndConditions       core/chessEngine.py:632-651   (mate/stalemate/draw50 only;
 *                                  the repetition dictionary lives in the host shim)
 *   - isDraw (only-kings clause)  core/chessEngine.py:21-33
 *   - encode_board / encode_move  ai/ai.py:17-57
 * The quirks of that file (SURVEY.md §8a-Q) are reproduced on purpose.
 *
 * Parity pinning: tests/test_oracle_golden.py checks this file against fixtures generated
 * by running the UNMODIFIED Python reference in the build container
 * (oracle/gen_golden.py -> tests/golden/).  The MCTS part (kvo_mcts_*) has no reference
 * counterpart ("parity unpinned" — the reference has no tree search); it is the
 * executable specification of SPEC.md §MCTS.
 */
#include <stdint.h>
#include <string.h>
#include <stdlib.h>
#include <math.h>
#include "../include/kv_detmath.h"

#define KVO_API __attribute__((visibility("default")))

/* piece codes: 0 empty, 1+PIECE_TO_INDEX (ai/ai.py:7-10): wK wQ wR wB wN wp bK bQ bR bB bN bp */
enum { EMPTY = 0, WK = 1, WQ, WR, WB, WN, WP, BK, BQ, BR, BB, BN, BP };
enum { T_K = 0, T_Q, T_R, T_B, T_N, T_P };

#define IS_WHITE(p) ((p) >= WK && (p) <= WP)
#define IS_BLACK(p) ((p) >= BK)
#define PTYPE(p) (((p) - 1) % 6)

/* moved-flag bits (core/chessEngine.py:66-71) */
enum { F_WK = 1, F_BK = 2, F_WRK = 4, F_WRQ = 8, F_BRK = 16, F_BRQ = 32 };
/* move flags */
enum { MF_EP = 1, MF_CASTLE = 2, MF_PROMO = 4 };
/* result flags of getValidMoves */
enum { RF_CHECKMATE = 1, RF_STALEMATE = 2, RF_DRAW50 = 4, RF_E3_CHECK = 8, RF_ONLY_KINGS = 16,
       RF_STATE_MUTATED = 32, RF_OVERFLOW = 64 };

typedef struct {
    uint8_t board[64];      /* index = row*8+col, row 0 = rank 8 */
    uint8_t white_to_move;
    uint8_t wk_sq, bk_sq;   /* whiteKingLocation / blackKingLocation (independent of the board) */
    uint8_t moved;          /* F_* bits */
    int8_t ep_sq;           /* enPassantPossible, -1 = () */
    uint8_t pad[3];
    uint32_t clock;         /* halfMoveClock */
} kvo_state;

typedef struct {
    uint8_t from, to, flags;
    uint8_t piece_moved, piece_captured;
} kvo_move;

#define KVO_MAX_MOVES 512

typedef struct {
    kvo_move m[KVO_MAX_MOVES];
    int n;
} movelist;

typedef struct {
    int r, c, dr, dc;
} ray4;

/* ------------------------------------------------------------------------------------------ */

KVO_API void kvo_init_start(kvo_state *s) {
    static const uint8_t back_b[8] = { BR, BN, BB, BQ, BK, BB, BN, BR };
    static const uint8_t back_w[8] = { WR, WN, WB, WQ, WK, WB, WN, WR };
    memset(s, 0, sizeof(*s));
    for (int c = 0; c < 8; c++) {
        s->board[0 * 8 + c] = back_b[c];
        s->board[1 * 8 + c] = BP;
        s->board[6 * 8 + c] = WP;
        s->board[7 * 8 + c] = back_w[c];
    }
    s->white_to_move = 1;
    s->wk_sq = 7 * 8 + 4;
    s->bk_sq = 0 * 8 + 4;
    s->ep_sq = -1;
}

static inline int is_ally(const kvo_state *s, uint8_t p) {
    return s->white_to_move ? IS_WHITE(p) : IS_BLACK(p);
}
static inline int is_enemy(const kvo_state *s, uint8_t p) {
    return s->white_to_move ? IS_BLACK(p) : IS_WHITE(p);
}

static inline void push_move(const kvo_state *s, movelist *ml, int from, int to, int flags) {
    /* Move.__init__, core/chessEngine.py:693-713 */
    if (ml->n >= KVO_MAX_MOVES) return;
    kvo_move *m = &ml->m[ml->n++];
    m->from = (uint8_t)from;
    m->to = (uint8_t)to;
    m->piece_moved = s->board[from];
    m->piece_captured = s->board[to];
    m->flags = (uint8_t)flags;
    if (flags & MF_EP) m->piece_captured = (m->piece_moved == WP) ? BP : WP;
    if ((m->piece_moved == WP && (to >> 3) == 0) || (m->piece_moved == BP && (to >> 3) == 7))
        m->flags |= MF_PROMO;
}

typedef struct {
    kvo_state *s;
    int inside_sua; /* insideSquareUnderAttack, core/chessEngine.py:61 */
} ctx_t;

static int square_under_attack(ctx_t *cx, int r, int c);
static void gen_all(ctx_t *cx, movelist *ml, const ray4 *pins, int npins);

/* getPawnMoves, core/chessEngine.py:447-472.  has_pin: pinDirection given. */
static void gen_pawn(ctx_t *cx, int r, int c, movelist *ml, int has_pin, int pr, int pc) {
    kvo_state *s = cx->s;
    int ma = s->white_to_move ? -1 : 1;
    int start_row = s->white_to_move ? 6 : 1;
    if (!has_pin || (pr == ma && pc == 0)) {
        int r1 = r + ma;
        if (r1 >= 0 && r1 < 8 && s->board[r1 * 8 + c] == EMPTY) {
            push_move(s, ml, r * 8 + c, r1 * 8 + c, 0);
            if (r == start_row && s->board[(r + 2 * ma) * 8 + c] == EMPTY)
                push_move(s, ml, r * 8 + c, (r + 2 * ma) * 8 + c, 0);
        }
    }
    for (int k = 0; k < 2; k++) {
        int dc = k ? 1 : -1;
        if (c + dc < 0 || c + dc >= 8) continue;
        if (has_pin && !(pr == ma && pc == dc)) continue;
        int r1 = r + ma;
        if (r1 < 0 || r1 >= 8) continue;
        int t = r1 * 8 + c + dc;
        if (is_enemy(s, s->board[t]))
            push_move(s, ml, r * 8 + c, t, 0);
        else if (t == s->ep_sq)
            push_move(s, ml, r * 8 + c, t, MF_EP);
    }
}

/* getRookMoves :477-494 / getBishopMoves :516-531 share the same walk */
static void gen_slider(ctx_t *cx, int r, int c, movelist *ml, const int (*dirs)[2]) {
    kvo_state *s = cx->s;
    for (int k = 0; k < 4; k++) {
        for (int i = 1; i < 8; i++) {
            int er = r + dirs[k][0] * i, ec = c + dirs[k][1] * i;
            if (er < 0 || er >= 8 || ec < 0 || ec >= 8) break;
            uint8_t p = s->board[er * 8 + ec];
            if (p == EMPTY) {
                push_move(s, ml, r * 8 + c, er * 8 + ec, 0);
            } else if (is_enemy(s, p)) {
                push_move(s, ml, r * 8 + c, er * 8 + ec, 0);
                break;
            } else {
                break;
            }
        }
    }
}
static const int ROOK_DIRS[4][2] = { { -1, 0 }, { 1, 0 }, { 0, -1 }, { 0, 1 } };
static const int BISHOP_DIRS[4][2] = { { -1, -1 }, { -1, 1 }, { 1, -1 }, { 1, 1 } };

/* getKnightMoves :500-512 */
static void gen_knight(ctx_t *cx, int r, int c, movelist *ml) {
    static const int km[8][2] = { { -2, -1 }, { -1, -2 }, { -2, 1 }, { -1, 2 },
                                  { 1, -2 },  { 2, -1 },  { 1, 2 },  { 2, 1 } };
    kvo_state *s = cx->s;
    for (int k = 0; k < 8; k++) {
        int er = r + km[k][0], ec = c + km[k][1];
        if (er < 0 || er >= 8 || ec < 0 || ec >= 8) continue;
        uint8_t p = s->board[er * 8 + ec];
        if (p == EMPTY || !is_ally(s, p)) push_move(s, ml, r * 8 + c, er * 8 + ec, 0);
    }
}

/* getCastleMoves :575-601 */
static void gen_castle(ctx_t *cx, int r, int c, movelist *ml) {
    kvo_state *s = cx->s;
    if (square_under_attack(cx, r, c)) return;
    if (s->white_to_move) {
        if (s->wk_sq != 60 || (s->moved & F_WK)) return;
        if (!(s->moved & F_WRK) && s->board[61] == EMPTY && s->board[62] == EMPTY)
            if (!square_under_attack(cx, 7, 5) && !square_under_attack(cx, 7, 6))
                if (s->board[63] == WR) push_move(s, ml, 60, 62, MF_CASTLE);
        if (!(s->moved & F_WRQ) && s->board[57] == EMPTY && s->board[58] == EMPTY && s->board[59] == EMPTY)
            if (!square_under_attack(cx, 7, 2) && !square_under_attack(cx, 7, 3))
                if (s->board[56] == WR) push_move(s, ml, 60, 58, MF_CASTLE);
    } else {
        if (s->bk_sq != 4 || (s->moved & F_BK)) return;
        if (!(s->moved & F_BRK) && s->board[5] == EMPTY && s->board[6] == EMPTY)
            if (!square_under_attack(cx, 0, 5) && !square_under_attack(cx, 0, 6))
                if (s->board[7] == BR) push_move(s, ml, 4, 6, MF_CASTLE);
        if (!(s->moved & F_BRQ) && s->board[1] == EMPTY && s->board[2] == EMPTY && s->board[3] == EMPTY)
            if (!square_under_attack(cx, 0, 2) && !square_under_attack(cx, 0, 3))
                if (s->board[0] == BR) push_move(s, ml, 4, 2, MF_CASTLE);
    }
}

/* getKingMoves :543-573.  NOTE the restore at :564 copies the placed king back to (r,c):
 * when (r,c) did not hold a king (stale king location in the >=2-checks branch, :315) this
 * permanently writes a king there.  Reproduced. */
static void gen_king(ctx_t *cx, int r, int c, movelist *ml) {
    static const int kd[8][2] = { { -1, -1 }, { -1, 0 }, { -1, 1 }, { 0, -1 },
                                  { 0, 1 },   { 1, -1 }, { 1, 0 },  { 1, 1 } };
    kvo_state *s = cx->s;
    for (int k = 0; k < 8; k++) {
        int er = r + kd[k][0], ec = c + kd[k][1];
        if (er < 0 || er >= 8 || ec < 0 || ec >= 8) continue;
        uint8_t p = s->board[er * 8 + ec];
        if (p == EMPTY || !is_ally(s, p)) {
            uint8_t orig = p;
            s->board[r * 8 + c] = EMPTY;
            s->board[er * 8 + ec] = s->white_to_move ? WK : BK;
            uint8_t orig_loc = s->white_to_move ? s->wk_sq : s->bk_sq;
            if (s->white_to_move) s->wk_sq = (uint8_t)(er * 8 + ec);
            else s->bk_sq = (uint8_t)(er * 8 + ec);
            int in_check = square_under_attack(cx, er, ec);
            s->board[r * 8 + c] = s->board[er * 8 + ec];
            s->board[er * 8 + ec] = orig;
            if (s->white_to_move) s->wk_sq = orig_loc;
            else s->bk_sq = orig_loc;
            if (!in_check) push_move(s, ml, r * 8 + c, er * 8 + ec, 0);
        }
    }
    gen_castle(cx, r, c, ml);
}

static void gen_piece(ctx_t *cx, int type, int r, int c, movelist *ml) {
    switch (type) {
    case T_R: gen_slider(cx, r, c, ml, ROOK_DIRS); break;
    case T_B: gen_slider(cx, r, c, ml, BISHOP_DIRS); break;
    case T_Q:
        gen_slider(cx, r, c, ml, ROOK_DIRS);
        gen_slider(cx, r, c, ml, BISHOP_DIRS);
        break;
    case T_N: gen_knight(cx, r, c, ml); break;
    case T_K: gen_king(cx, r, c, ml); break;
    default: break;
    }
}

/* addPieceMovesConsideringPins :604-630 */
static void add_piece_moves(ctx_t *cx, int type, int r, int c, movelist *ml, const ray4 *pins, int npins) {
    int pinned = 0, pr = 0, pc = 0;
    for (int i = npins - 1; i >= 0; i--) {
        if (pins[i].r == r && pins[i].c == c) {
            pinned = 1;
            pr = pins[i].dr;
            pc = pins[i].dc;
            break;
        }
    }
    if (pinned) {
        if (type == T_N) return;
        movelist tmp;
        tmp.n = 0;
        if (type == T_P) gen_pawn(cx, r, c, &tmp, 1, pr, pc);
        else gen_piece(cx, type, r, c, &tmp);
        for (int i = 0; i < tmp.n; i++) {
            int mr = (tmp.m[i].to >> 3) - r, mc = (tmp.m[i].to & 7) - c;
            if (mr * pc == mc * pr && ml->n < KVO_MAX_MOVES) ml->m[ml->n++] = tmp.m[i];
        }
    } else {
        if (type == T_P) gen_pawn(cx, r, c, ml, 0, 0, 0);
        else gen_piece(cx, type, r, c, ml);
    }
}

/* getAllPossibleMoves :433-441 */
static void gen_all(ctx_t *cx, movelist *ml, const ray4 *pins, int npins) {
    kvo_state *s = cx->s;
    ml->n = 0;
    for (int r = 0; r < 8; r++)
        for (int c = 0; c < 8; c++) {
            uint8_t p = s->board[r * 8 + c];
            if (p != EMPTY && is_ally(s, p)) add_piece_moves(cx, PTYPE(p), r, c, ml, pins, npins);
        }
}

/* squareUnderAttack :400-415 */
static int square_under_attack(ctx_t *cx, int r, int c) {
    if (cx->inside_sua) return 0;
    cx->inside_sua = 1;
    kvo_state *s = cx->s;
    uint8_t orig = s->white_to_move;
    s->white_to_move = !orig;
    movelist opp;
    gen_all(cx, &opp, NULL, 0);
    s->white_to_move = orig;
    cx->inside_sua = 0;
    int t = r * 8 + c;
    for (int i = 0; i < opp.n; i++)
        if (opp.m[i].to == t) return 1;
    return 0;
}

/* checkForPinsAndChecks :325-383 */
static int pins_and_checks(const kvo_state *s, ray4 *pins, int *npins, ray4 *checks, int *nchecks) {
    static const int dirs[8][2] = { { -1, 0 }, { 0, -1 }, { 1, 0 }, { 0, 1 },
                                    { -1, -1 }, { -1, 1 }, { 1, -1 }, { 1, 1 } };
    static const int kn[7][2] = { { -2, -1 }, { -1, -2 }, { -1, 2 }, { 1, -2 }, { 2, -1 }, { 1, 2 }, { 2, 1 } };
    int in_check = 0;
    *npins = 0;
    *nchecks = 0;
    int ksq = s->white_to_move ? s->wk_sq : s->bk_sq;
    int kr = ksq >> 3, kc = ksq & 7;
    int enemy_white = !s->white_to_move;
    for (int d = 0; d < 8; d++) {
        int have_pin = 0;
        ray4 pp = { 0, 0, 0, 0 };
        for (int i = 1; i < 8; i++) {
            int er = kr + dirs[d][0] * i, ec = kc + dirs[d][1] * i;
            if (er < 0 || er >= 8 || ec < 0 || ec >= 8) break;
            uint8_t p = s->board[er * 8 + ec];
            if (p == EMPTY) continue;
            if (is_ally(s, p)) {
                if (!have_pin) {
                    have_pin = 1;
                    pp.r = er; pp.c = ec; pp.dr = dirs[d][0]; pp.dc = dirs[d][1];
                } else {
                    break;
                }
            } else {
                int t = PTYPE(p);
                int orth = d < 4;
                int pawn_dir_ok = enemy_white ? (dirs[d][0] == 1 && dirs[d][1] != 0)
                                              : (dirs[d][0] == -1 && dirs[d][1] != 0);
                if ((orth && (t == T_R || t == T_Q)) || (!orth && (t == T_B || t == T_Q)) ||
                    (i == 1 && t == T_P && pawn_dir_ok)) {
                    if (!have_pin) {
                        in_check = 1;
                        checks[*nchecks].r = er; checks[*nchecks].c = ec;
                        checks[*nchecks].dr = dirs[d][0]; checks[*nchecks].dc = dirs[d][1];
                        (*nchecks)++;
                    } else {
                        pins[(*npins)++] = pp;
                    }
                }
                break;
            }
        }
    }
    for (int k = 0; k < 7; k++) {
        int er = kr + kn[k][0], ec = kc + kn[k][1];
        if (er < 0 || er >= 8 || ec < 0 || ec >= 8) continue;
        uint8_t p = s->board[er * 8 + ec];
        if (p != EMPTY && is_enemy(s, p) && PTYPE(p) == T_N) {
            in_check = 1;
            checks[*nchecks].r = er; checks[*nchecks].c = ec;
            checks[*nchecks].dr = kn[k][0]; checks[*nchecks].dc = kn[k][1];
            (*nchecks)++;
        }
    }
    return in_check;
}

static int only_kings(const kvo_state *s) {
    for (int i = 0; i < 64; i++)
        if (s->board[i] != EMPTY && s->board[i] != WK && s->board[i] != BK) return 0;
    return 1;
}

/* getValidMoves :277-321.  Returns the number of moves; *rflags gets RF_* bits. */
static int valid_moves(kvo_state *s, movelist *out, int *rflags) {
    ctx_t cx = { s, 0 };
    ray4 pins[8], checks[16];
    int npins, nchecks;
    kvo_state before = *s;
    int in_check = pins_and_checks(s, pins, &npins, checks, &nchecks);
    int ksq = s->white_to_move ? s->wk_sq : s->bk_sq;
    int kr = ksq >> 3, kc = ksq & 7;
    out->n = 0;
    if (in_check) {
        if (nchecks == 1) {
            movelist all;
            gen_all(&cx, &all, pins, npins);
            uint64_t valid = 0;
            ray4 ck = checks[0];
            uint8_t checker = s->board[ck.r * 8 + ck.c];
            if (PTYPE(checker) == T_N) {
                valid = 1ull << (ck.r * 8 + ck.c);
            } else {
                for (int i = 1; i < 8; i++) {
                    int r = kr + ck.dr * i, c = kc + ck.dc * i;
                    /* the reference appends tuples without bounds checks; the walk always
                       terminates at the checker square, which is on the board */
                    if (r >= 0 && r < 8 && c >= 0 && c < 8) valid |= 1ull << (r * 8 + c);
                    if (r == ck.r && c == ck.c) break;
                }
            }
            for (int i = 0; i < all.n; i++) {
                kvo_move *m = &all.m[i];
                if (m->piece_moved != EMPTY && PTYPE(m->piece_moved) == T_K) {
                    if (!square_under_attack(&cx, m->to >> 3, m->to & 7)) out->m[out->n++] = *m;
                } else if ((valid >> m->to) & 1) {
                    out->m[out->n++] = *m;
                }
            }
        } else {
            gen_king(&cx, kr, kc, out);
        }
    } else {
        gen_all(&cx, out, pins, npins);
    }
    int f = 0;
    if (in_check) f |= RF_E3_CHECK;
    /* checkForEndConditions :632-651 (repetition handled by the host shim) */
    if (out->n == 0) {
        if (square_under_attack(&cx, ksq >> 3, ksq & 7)) f |= RF_CHECKMATE;
        else f |= RF_STALEMATE;
    } else if (s->clock >= 100) {
        f |= RF_DRAW50;
    }
    if (only_kings(s)) f |= RF_ONLY_KINGS;
    if (memcmp(before.board, s->board, 64) != 0) f |= RF_STATE_MUTATED;
    *rflags = f;
    return out->n;
}

/* makeMove :127-197 (no legality check).  promo_type: T_Q by default (Move.promotionChoice). */
static void make_move(kvo_state *s, int from, int to, int flags, int promo_type) {
    uint8_t pm = s->board[from];
    uint8_t pcap = s->board[to];
    if (flags & MF_EP) pcap = (pm == WP) ? BP : WP;
    int sr = from >> 3, sc = from & 7, er = to >> 3, ec = to & 7;
    s->board[from] = EMPTY;
    s->board[to] = pm;
    if (pm == WK) s->moved |= F_WK;
    else if (pm == BK) s->moved |= F_BK;
    else if (pm == WR) {
        if (from == 56) s->moved |= F_WRQ;
        else if (from == 63) s->moved |= F_WRK;
    } else if (pm == BR) {
        if (from == 0) s->moved |= F_BRQ;
        else if (from == 7) s->moved |= F_BRK;
    }
    if (flags & MF_EP) s->board[sr * 8 + ec] = EMPTY;
    if (flags & MF_CASTLE) {
        if (ec - sc == 2) {
            if (ec + 1 < 8) { /* the reference would raise IndexError otherwise */
                s->board[er * 8 + ec - 1] = s->board[er * 8 + ec + 1];
                s->board[er * 8 + ec + 1] = EMPTY;
            }
        } else {
            if (ec - 2 >= 0 && ec + 1 < 8) {
                s->board[er * 8 + ec + 1] = s->board[er * 8 + ec - 2];
                s->board[er * 8 + ec - 2] = EMPTY;
            }
        }
    }
    if (pm != EMPTY && PTYPE(pm) == T_P && abs(sr - er) == 2) s->ep_sq = (int8_t)(((sr + er) / 2) * 8 + sc);
    else s->ep_sq = -1;
    if (pcap != EMPTY) s->clock = 0; /* 'P' typo at :178 — pawn moves never reset */
    else s->clock += 1;
    s->white_to_move = !s->white_to_move;
    if (pm == WK) s->wk_sq = (uint8_t)to;
    else if (pm == BK) s->bk_sq = (uint8_t)to;
    if (flags & MF_PROMO) s->board[to] = (uint8_t)((IS_WHITE(pm) ? 1 : 7) + promo_type);
}

/* ------------------------------------------------------------------------------------------
 * Packed 128-byte board line (the device layout, include/kv_b200.h):
 *   w[0..11]  bitboards in PIECE_TO_INDEX order, bit = row*8+col
 *   w[12]     meta: bit0 whiteToMove | bits1-6 moved flags | bits8-14 ep (64=none)
 *             | bits16-21 wk_sq | bits24-29 bk_sq | bits32-47 clock
 *   w[13..15] reserved (0)
 * ------------------------------------------------------------------------------------------ */
KVO_API void kvo_pack(const kvo_state *s, uint64_t *w) {
    memset(w, 0, 16 * sizeof(uint64_t));
    for (int i = 0; i < 64; i++)
        if (s->board[i]) w[s->board[i] - 1] |= 1ull << i;
    uint64_t ep = s->ep_sq < 0 ? 64 : (uint64_t)s->ep_sq;
    uint32_t clk = s->clock > 0xFFFF ? 0xFFFF : s->clock;
    w[12] = (uint64_t)(s->white_to_move & 1) | ((uint64_t)(s->moved & 63) << 1) | (ep << 8) |
            ((uint64_t)s->wk_sq << 16) | ((uint64_t)s->bk_sq << 24) | ((uint64_t)clk << 32);
}

KVO_API void kvo_unpack(const uint64_t *w, kvo_state *s) {
    memset(s, 0, sizeof(*s));
    for (int p = 0; p < 12; p++)
        for (int i = 0; i < 64; i++)
            if ((w[p] >> i) & 1) s->board[i] = (uint8_t)(p + 1);
    uint64_t m = w[12];
    s->white_to_move = m & 1;
    s->moved = (m >> 1) & 63;
    int ep = (m >> 8) & 127;
    s->ep_sq = ep >= 64 ? -1 : (int8_t)ep;
    s->wk_sq = (m >> 16) & 63;
    s->bk_sq = (m >> 24) & 63;
    s->clock = (m >> 32) & 0xFFFF;
}

static inline uint16_t pack_move(const kvo_move *m) {
    return (uint16_t)(m->from | (m->to << 6) | ((m->flags & 7) << 12));
}

/* Batched API over packed lines (same shapes as the device C-ABI). */
KVO_API void kvo_movegen(uint64_t *lines, int n, uint16_t *moves, int stride, int32_t *counts, int32_t *flags) {
    for (int i = 0; i < n; i++) {
        kvo_state s;
        movelist ml;
        int f;
        kvo_unpack(lines + 16 * (size_t)i, &s);
        int cnt = valid_moves(&s, &ml, &f);
        if (cnt > stride) { f |= RF_OVERFLOW; }
        for (int k = 0; k < cnt && k < stride; k++) moves[(size_t)i * stride + k] = pack_move(&ml.m[k]);
        counts[i] = cnt;
        flags[i] = f;
        if (f & RF_STATE_MUTATED) kvo_pack(&s, lines + 16 * (size_t)i);
    }
}

KVO_API void kvo_make_moves(uint64_t *lines, int n, const uint16_t *mv) {
    for (int i = 0; i < n; i++) {
        kvo_state s;
        kvo_unpack(lines + 16 * (size_t)i, &s);
        make_move(&s, mv[i] & 63, (mv[i] >> 6) & 63, (mv[i] >> 12) & 7, T_Q);
        kvo_pack(&s, lines + 16 * (size_t)i);
    }
}

KVO_API int kvo_square_under_attack(const uint64_t *line, int r, int c) {
    kvo_state s;
    kvo_unpack(line, &s);
    ctx_t cx = { &s, 0 };
    return square_under_attack(&cx, r, c);
}

KVO_API int kvo_in_check(const uint64_t *line) {
    kvo_state s;
    kvo_unpack(line, &s);
    ctx_t cx = { &s, 0 };
    int k = s.white_to_move ? s.wk_sq : s.bk_sq;
    return square_under_attack(&cx, k >> 3, k & 7);
}

/* perft: copy-make DFS over getValidMoves/makeMove with bulk counting at depth 1.
 * out[0] nodes, out[1] captures, out[2] ep, out[3] castles, out[4] promos (of leaf moves),
 * out[5] order digest: FNV-1a-64 over (from,to,flags) bytes of every move list visited, in DFS order. */
#define FNV_OFFSET 0xcbf29ce484222325ull
#define FNV_PRIME 0x100000001b3ull

static void perft_rec(const kvo_state *s, int depth, uint64_t *out) {
    kvo_state cur = *s;
    movelist ml;
    int f;
    int n = valid_moves(&cur, &ml, &f);
    uint64_t h = out[5];
    for (int i = 0; i < n; i++) {
        h = (h ^ ml.m[i].from) * FNV_PRIME;
        h = (h ^ ml.m[i].to) * FNV_PRIME;
        h = (h ^ (ml.m[i].flags & 7)) * FNV_PRIME;
    }
    out[5] = h;
    if (depth == 1) {
        out[0] += (uint64_t)n;
        for (int i = 0; i < n; i++) {
            if (ml.m[i].piece_captured != EMPTY) out[1]++;
            if (ml.m[i].flags & MF_EP) out[2]++;
            if (ml.m[i].flags & MF_CASTLE) out[3]++;
            if (ml.m[i].flags & MF_PROMO) out[4]++;
        }
        return;
    }
    for (int i = 0; i < n; i++) {
        kvo_state child = cur;
        make_move(&child, ml.m[i].from, ml.m[i].to, ml.m[i].flags, T_Q);
        perft_rec(&child, depth - 1, out);
    }
}

KVO_API void kvo_perft(const uint64_t *line, int depth, uint64_t *out6) {
    kvo_state s;
    kvo_unpack(line, &s);
    memset(out6, 0, 6 * sizeof(uint64_t));
    out6[5] = FNV_OFFSET;
    if (depth <= 0) { out6[0] = 1; return; }
    perft_rec(&s, depth, out6);
}

/* perft2: the quantities the GPU perft driver reports (include/kv_b200.h, kv_perft).  The GPU frontier is an
 * unordered multiset, so the order digest is an order-independent SUM of per-list hashes, each seeded by the
 * hash of the path that leads to the list: still sensitive to the order of moves inside every list.
 * out[0] nodes, [1] captures, [2] ep, [3] castles, [4] promos, [5] digest, [6] movegen calls, [7] 0. */
static uint64_t mix64(uint64_t x) {
    x ^= x >> 30;
    x *= 0xbf58476d1ce4e5b9ull;
    x ^= x >> 27;
    x *= 0x94d049bb133111ebull;
    x ^= x >> 31;
    return x;
}

static void perft2_rec(const kvo_state *s, int depth, uint64_t path, uint64_t *out) {
    kvo_state cur = *s;
    movelist ml;
    int f;
    int n = valid_moves(&cur, &ml, &f);
    if (n > 256) n = 256;
    out[6]++;
    for (int k = 0; k < n; k++)
        out[5] += mix64(path + (uint64_t)(k + 1) * 0x9E3779B97F4A7C15ull + ((uint64_t)pack_move(&ml.m[k]) << 32));
    if (depth == 1) {
        out[0] += (uint64_t)n;
        for (int i = 0; i < n; i++) {
            if (ml.m[i].piece_captured != EMPTY) out[1]++;
            if (ml.m[i].flags & MF_EP) out[2]++;
            if (ml.m[i].flags & MF_CASTLE) out[3]++;
            if (ml.m[i].flags & MF_PROMO) out[4]++;
        }
        return;
    }
    for (int k = 0; k < n; k++) {
        kvo_state child = cur;
        make_move(&child, ml.m[k].from, ml.m[k].to, ml.m[k].flags, T_Q);
        perft2_rec(&child, depth - 1, mix64(path ^ ((uint64_t)(k + 1) * 0xD6E8FEB86659FD93ull)), out);
    }
}

KVO_API void kvo_perft2(const uint64_t *line, int depth, uint64_t *out8) {
    kvo_state s;
    kvo_unpack(line, &s);
    memset(out8, 0, 8 * sizeof(uint64_t));
    perft2_rec(&s, depth, 0, out8);
}

/* encode_board, ai/ai.py:17-41 (list branch): float32 [12,8,8] one-hot */
KVO_API void kvo_encode(const uint64_t *lines, int n, float *planes) {
    for (int i = 0; i < n; i++)
        for (int p = 0; p < 12; p++)
            for (int sq = 0; sq < 64; sq++)
                planes[((size_t)i * 12 + p) * 64 + sq] = (float)((lines[16 * (size_t)i + p] >> sq) & 1);
}

/* encode_move ai/ai.py:51-57 */
KVO_API int kvo_move_index(uint16_t mv) { return (mv & 63) * 64 + ((mv >> 6) & 63); }


/* ==========================================================================================================
 * MCTS oracle — "parity unpinned": the reference has no tree search (SURVEY.md fact 1), so this sequential PUCT
 * over the pinned rules engine above IS the specification (DESIGN.md §MCTS) that the GPU tree kernels must match
 * bit-for-bit (visit counts, W sums, chosen moves), given identical evaluator outputs and seeds.
 * Evaluator modes: 0 = deterministic hash evaluator (also implemented on the device: whole-pipeline parity,
 * including softmax / Dirichlet arithmetic), 1 = replay of the values and priors the device engine recorded
 * for its own network evaluations (tree-logic parity "given identical net outputs").
 * ========================================================================================================== */
typedef struct {
    int32_t sims;        /* simulations per move (the first one expands the root) */
    int32_t edge_cap;    /* edges per game tree; an expansion that does not fit becomes a terminal draw */
    int32_t temp_plies;  /* plies < temp_plies sample the move from the visit counts, later plies take the argmax */
    int32_t max_plies;   /* game is a draw when this many plies were played */
    float c_puct, dir_alpha, dir_eps;
    int32_t inflight;    /* K simulations in flight per wave (0 or 1: sequential search; > 1: virtual loss) */
    uint64_t seed;
    float resign_thr;          /* scripts/self_play.py:185: value < thr (reference -0.7) ... */
    int32_t resign_min_plies;  /* ... once more than this many plies were played (reference 15); < 0: never */
    int32_t root_mix;          /* 1: root priors by scripts/self_play.py:150-167 (all 4096 indices), 0: legal moves only */
    int32_t pad;
} kvo_mcts_cfg;
#define POLICY_N 4096

typedef struct {
    kvo_state st;
    int32_t first_edge, n_edges;
    uint32_t N;          /* 1 + completed simulations through the node */
    uint32_t VL;         /* virtual visits: simulations of the current wave that went through and are not backed up */
    int32_t term;
    int32_t pending;     /* created in the current wave, priors not delivered yet */
    float val;           /* terminal value, or the evaluator's value, from the node's side to move */
} onode;
typedef struct {
    float P, W;
    uint32_t N, VL;
    int32_t child;
    uint16_t mv;
} oedge;

static uint64_t pos_hash(const uint64_t *bb) {
    uint64_t h = 0x243F6A8885A308D3ull;
    for (int p = 0; p < 12; p++) h = kvd_mix64(h ^ (bb[p] + (uint64_t)(p + 1) * 0x9E3779B97F4A7C15ull));
    return h;
}

/* hash evaluator: logit of move index idx and the white-perspective value */
static float hash_logit(uint64_t ph, int idx) { return (float)kvd_rand24(ph, (uint64_t)idx, 1, 0) * (4.0f / 16777216.0f) - 2.0f; }
static float hash_value(uint64_t ph) { return (float)kvd_rand24(ph, 4096, 2, 0) * (2.0f / 16777216.0f) - 1.0f; }

typedef struct {
    /* replay inputs (device tree dump), NULL in hash mode */
    const float *rep_node_val;
    const int32_t *rep_node_first;
    const float *rep_edge_P;
} replay_t;

/* e[k].P holds the legal moves' logits (mx = their maximum): softmax over the legal moves, and at the root the Dirichlet
 * noise over the legal moves (DESIGN.md 4.3; the arithmetic and its order are the device's, mcts_expand_warp) */
static void priors_from_logits(const kvo_mcts_cfg *cfg, oedge *e, int n, float mx, int is_root, uint64_t game_id, int ply) {
    float sum = 0.0f;
    for (int k = 0; k < n; k++) {
        e[k].P = kvd_expf(e[k].P - mx);
        sum = sum + e[k].P;
    }
    for (int k = 0; k < n; k++) e[k].P = e[k].P / sum;
    if (is_root && cfg->dir_eps > 0.0f) {
        float gs = 0.0f;
        for (int k = 0; k < n; k++) {
            e[k].W = kvd_gamma_small(cfg->dir_alpha, cfg->seed, game_id, (uint64_t)ply * 256 + (uint64_t)k);
            gs = gs + e[k].W;
        }
        for (int k = 0; k < n; k++) {
            const float eta = e[k].W / gs;
            e[k].P = (1.0f - cfg->dir_eps) * e[k].P + cfg->dir_eps * eta;
            e[k].W = 0.0f;
        }
    }
}

/* priors and value of a freshly expanded (non-terminal) leaf: replayed device outputs, or the hash evaluator with the
 * softmax / root-noise arithmetic of DESIGN.md 4.3 */
static void evaluate_leaf(const kvo_mcts_cfg *cfg, onode *nd, oedge *e, int leaf, uint64_t game_id, int ply,
                          const replay_t *rep) {
    const int n = nd->n_edges;
    if (rep && rep->rep_node_val) {
        nd->val = rep->rep_node_val[leaf];
        for (int k = 0; k < n; k++) e[k].P = rep->rep_edge_P[rep->rep_node_first[leaf] + k];
        return;
    }
    uint64_t w[16];
    kvo_pack(&nd->st, w);
    const uint64_t ph = pos_hash(w);
    float mx = 0.0f;
    for (int k = 0; k < n; k++) {
        e[k].P = hash_logit(ph, kvo_move_index(e[k].mv));
        if (k == 0 || e[k].P > mx) mx = e[k].P;
    }
    if (leaf == 0 && cfg->root_mix) {
        /* scripts/self_play.py:150-167: policy = softmax over ALL 4096 logits; noise = Dirichlet(alpha) over all 4096
         * indices; policy = (1-eps) policy + eps noise; the legal entries renormalised (:159-166).  Reductions in the
         * order of the device warp: lane-strided partials (lane = index mod 32), then an xor butterfly. */
        float part[32];
        for (int l = 0; l < 32; l++) part[l] = -3.0e38f;
        for (int i = 0; i < POLICY_N; i++) {
            const float lg = hash_logit(ph, i);
            if (lg > part[i & 31]) part[i & 31] = lg;
        }
        float mxa = part[0];
        for (int l = 1; l < 32; l++) if (part[l] > mxa) mxa = part[l];
        for (int l = 0; l < 32; l++) part[l] = 0.0f;
        for (int i = 0; i < POLICY_N; i++) part[i & 31] = part[i & 31] + kvd_expf(hash_logit(ph, i) - mxa);
        for (int d = 16; d >= 1; d >>= 1) {
            float nx[32];
            for (int l = 0; l < 32; l++) nx[l] = part[l] + part[l ^ d];
            memcpy(part, nx, sizeof(nx));
        }
        const float z = part[0];
        for (int k = 0; k < n; k++) e[k].P = kvd_expf(e[k].P - mxa) / z;
        if (cfg->dir_eps > 0.0f) {
            const uint64_t key = (uint64_t)ply * POLICY_N;
            for (int l = 0; l < 32; l++) part[l] = 0.0f;
            for (int i = 0; i < POLICY_N; i++)
                part[i & 31] = part[i & 31] + kvd_gamma_small(cfg->dir_alpha, cfg->seed, game_id, key + (uint64_t)i);
            for (int d = 16; d >= 1; d >>= 1) {
                float nx[32];
                for (int l = 0; l < 32; l++) nx[l] = part[l] + part[l ^ d];
                memcpy(part, nx, sizeof(nx));
            }
            const float gsum = part[0];
            for (int k = 0; k < n; k++) {
                const float g = kvd_gamma_small(cfg->dir_alpha, cfg->seed, game_id, key + (uint64_t)kvo_move_index(e[k].mv));
                e[k].P = (1.0f - cfg->dir_eps) * e[k].P + cfg->dir_eps * (g / gsum);
            }
        }
        float sum = 0.0f;
        for (int k = 0; k < n; k++) sum = sum + e[k].P;
        for (int k = 0; k < n; k++) e[k].P = e[k].P / sum;
        const float vw0 = hash_value(ph);
        nd->val = nd->st.white_to_move ? vw0 : -vw0;
        return;
    }
    priors_from_logits(cfg, e, n, mx, leaf == 0, game_id, ply);
    const float vw = hash_value(ph);
    nd->val = nd->st.white_to_move ? vw : -vw;
}

/* backup of one simulation: the virtual visit taken at selection becomes the real one */
static void backup_path(onode *nodes, oedge *edges, const int *path_n, const int *path_e, int depth, float v) {
    for (int i = depth - 1; i >= 0; i--) {
        v = -v;
        edges[path_e[i]].W = edges[path_e[i]].W + v;
        edges[path_e[i]].N++;
        edges[path_e[i]].VL--;
        nodes[path_n[i]].N++;
        nodes[path_n[i]].VL--;
    }
}

/* the move of a finished search: index into the root's n edges (total = sum of their visit counts) */
static int choose_move(const kvo_mcts_cfg *cfg, const oedge *e, int n, uint64_t total, uint64_t game_id, int ply) {
    int pick = 0;
    if (total == 0) {
        /* sims == 1: sample from the (noisy) priors, the reference's own move rule (scripts/self_play.py:147-167) */
        const float u = kvd_u01(kvd_rand24(cfg->seed, game_id, (uint64_t)ply, 0xC0FFEEull));
        float sum = 0.0f;
        for (int k = 0; k < n; k++) sum = sum + e[k].P;
        const float thr = u * sum;
        float cum = 0.0f;
        pick = n - 1;
        for (int k = 0; k < n; k++) {
            cum = cum + e[k].P;
            if (cum > thr) { pick = k; break; }
        }
    } else if (ply < cfg->temp_plies) {
        const uint64_t r = ((uint64_t)kvd_rand24(cfg->seed, game_id, (uint64_t)ply, 0xC0FFEEull) * total) >> 24;
        uint64_t cum = 0;
        for (int k = 0; k < n; k++) {
            cum += e[k].N;
            if (cum > r) { pick = k; break; }
        }
    } else {
        for (int k = 1; k < n; k++)
            if (e[k].N > e[pick].N) pick = k;
    }
    return pick;
}

/* Optional copy of the whole tree at the end of a search (kvo_mcts_search_tree); NULL members are skipped. */
typedef struct {
    uint64_t *node_line;   /* [sims + 1][16] the node's line as stored after move generation (the evaluated position) */
    int32_t *node_i32;     /* [sims + 1][4]  terminal flag, first edge (-1 none), edge count, visits N */
    float *node_val;       /* [sims + 1]     terminal value or the evaluator's value, from the node's side to move */
    uint16_t *edge_mv;     /* [edge_cap]     move word */
    int32_t *edge_child;   /* [edge_cap]     child node, -1 unexpanded */
    float *edge_P, *edge_W;
    uint32_t *edge_N;
} tree_out_t;

/* Runs one search of cfg->sims simulations from `root`; returns the chosen move word (0xFFFF if the root has no
 * move).  Outputs: root move list, visit counts, W (bit patterns), number of nodes/edges created.
 *
 * The search proceeds in WAVES of up to K = cfg->inflight selections.  A selection descends by PUCT over
 * N + VL visits and W - VL value sums (virtual loss), marks its path with one virtual visit per edge and node, and
 * ends in (a) a terminal node or a new terminal leaf: backed up at once; (b) a new leaf that needs the evaluator:
 * it stays in flight until the end of the wave; (c) a leaf that is itself still in flight: the selection is undone
 * and the wave stops selecting.  At the end of the wave the in-flight leaves get their priors / values and are
 * backed up in selection order.  With K = 1 this is the plain sequential search (VL is 0 whenever a score is
 * computed). */
static int mcts_search(const kvo_mcts_cfg *cfg, const kvo_state *root, uint64_t game_id, int ply, const replay_t *rep,
                       uint16_t *root_moves, uint32_t *root_N, float *root_W, float *root_P, int *n_root,
                       int *out_nodes, int *out_edges, int *overflow, float *root_vwhite, const tree_out_t *tout) {
    const int S = cfg->sims;
    const int K = cfg->inflight > 1 ? cfg->inflight : 1;
    const size_t PL = (size_t)S + 2;   /* path stride */
    onode *nodes = (onode *)calloc((size_t)S + 1, sizeof(onode));
    oedge *edges = (oedge *)calloc((size_t)cfg->edge_cap, sizeof(oedge));
    int *path_e = (int *)malloc(sizeof(int) * PL * (size_t)K);
    int *path_n = (int *)malloc(sizeof(int) * PL * (size_t)K);
    int *pend_leaf = (int *)malloc(sizeof(int) * (size_t)K);
    int *pend_depth = (int *)malloc(sizeof(int) * (size_t)K);
    int n_nodes = 0, n_edges = 0, sims_done = 0;
    *overflow = 0;
    while (sims_done < S) {
        int n_pend = 0;
        for (int j = 0; j < K; j++) {
            if (sims_done + n_pend >= S) break;
            int *pe = path_e + PL * (size_t)n_pend, *pn = path_n + PL * (size_t)n_pend;
            int depth = 0, node = 0, leaf = -1, collided = 0;
            float v = 0.0f;
            kvo_state child_st;
            if (n_nodes == 0) {
                child_st = *root;
                leaf = 0;
            } else {
                for (;;) {
                    onode *nd = &nodes[node];
                    if (nd->pending) {
                        collided = 1;
                        break;
                    }
                    if (nd->term) {
                        v = nd->val;
                        nd->N++;
                        break;
                    }
                    const float sq = KVD_SQRTF((float)(nd->N + nd->VL));
                    int best = 0;
                    float bs = 0.0f;
                    for (int k = 0; k < nd->n_edges; k++) {
                        const oedge *e = &edges[nd->first_edge + k];
                        float sc = kvd_puct(e->W - (float)e->VL, e->N + e->VL, e->P, sq, cfg->c_puct);
                        if (k == 0 || sc > bs) { bs = sc; best = k; }
                    }
                    const int ei = nd->first_edge + best;
                    pn[depth] = node;
                    pe[depth] = ei;
                    depth++;
                    edges[ei].VL++;
                    nd->VL++;
                    if (edges[ei].child < 0) {
                        child_st = nd->st;
                        make_move(&child_st, edges[ei].mv & 63, (edges[ei].mv >> 6) & 63, (edges[ei].mv >> 12) & 7, T_Q);
                        leaf = n_nodes;
                        edges[ei].child = leaf;
                        break;
                    }
                    node = edges[ei].child;
                }
            }
            if (collided) {
                for (int i = depth - 1; i >= 0; i--) {
                    edges[pe[i]].VL--;
                    nodes[pn[i]].VL--;
                }
                break;   /* no more selections in this wave */
            }
            int in_flight = 0;
            if (leaf >= 0) {
                onode *nd = &nodes[leaf];
                movelist ml;
                int f;
                int n = valid_moves(&child_st, &ml, &f);   /* may rewrite child_st (getKingMoves restore quirk) */
                if (n > 256) n = 256;
                nd->st = child_st;
                nd->N = 1;
                nd->VL = 0;
                nd->first_edge = -1;
                nd->n_edges = 0;
                nd->pending = 0;
                n_nodes++;
                if (n == 0) {
                    nd->term = 1;
                    nd->val = (f & RF_CHECKMATE) ? -1.0f : 0.0f;
                } else if (f & RF_ONLY_KINGS) {
                    nd->term = 1;
                    nd->val = 0.0f;
                } else if (n_edges + n > cfg->edge_cap) {
                    nd->term = 1;
                    nd->val = 0.0f;
                    *overflow = 1;
                } else {
                    nd->term = 0;
                    nd->first_edge = n_edges;
                    nd->n_edges = n;
                    nd->pending = 1;
                    oedge *e = &edges[n_edges];
                    n_edges += n;
                    for (int k = 0; k < n; k++) {
                        e[k].mv = pack_move(&ml.m[k]);
                        e[k].N = 0;
                        e[k].VL = 0;
                        e[k].W = 0.0f;
                        e[k].P = 0.0f;
                        e[k].child = -1;
                    }
                    pend_leaf[n_pend] = leaf;
                    pend_depth[n_pend] = depth;
                    in_flight = 1;
                }
                v = nd->val;
            }
            if (in_flight) {
                n_pend++;
            } else {
                backup_path(nodes, edges, pn, pe, depth, v);
                sims_done++;
            }
        }
        /* end of the wave: the evaluator's answers arrive, then the backups in selection order */
        for (int j = 0; j < n_pend; j++) {
            onode *nd = &nodes[pend_leaf[j]];
            evaluate_leaf(cfg, nd, &edges[nd->first_edge], pend_leaf[j], game_id, ply, rep);
            nd->pending = 0;
        }
        for (int j = 0; j < n_pend; j++) {
            backup_path(nodes, edges, path_n + PL * (size_t)j, path_e + PL * (size_t)j, pend_depth[j],
                        nodes[pend_leaf[j]].val);
            sims_done++;
        }
    }
    int chosen = 0xFFFF;
    *n_root = 0;
    /* the evaluator's value of the root as the network returned it (white's perspective): what the resign rule reads */
    if (root_vwhite) *root_vwhite = n_nodes > 0 ? (nodes[0].st.white_to_move ? nodes[0].val : -nodes[0].val) : 0.0f;
    if (n_nodes > 0 && !nodes[0].term) {
        const int n = nodes[0].n_edges;
        const oedge *e = &edges[nodes[0].first_edge];
        *n_root = n;
        uint64_t total = 0;
        for (int k = 0; k < n; k++) {
            root_moves[k] = e[k].mv;
            root_N[k] = e[k].N;
            root_W[k] = e[k].W;
            root_P[k] = e[k].P;
            total += e[k].N;
        }
        chosen = e[choose_move(cfg, e, n, total, game_id, ply)].mv;
    }
    *out_nodes = n_nodes;
    *out_edges = n_edges;
    if (tout) {
        for (int i = 0; i < n_nodes; i++) {
            if (tout->node_line) kvo_pack(&nodes[i].st, tout->node_line + (size_t)i * 16);
            if (tout->node_i32) {
                int32_t *o = tout->node_i32 + (size_t)i * 4;
                o[0] = nodes[i].term;
                o[1] = nodes[i].first_edge;
                o[2] = nodes[i].n_edges;
                o[3] = (int32_t)nodes[i].N;
            }
            if (tout->node_val) tout->node_val[i] = nodes[i].val;
        }
        for (int i = 0; i < n_edges; i++) {
            if (tout->edge_mv) tout->edge_mv[i] = edges[i].mv;
            if (tout->edge_child) tout->edge_child[i] = edges[i].child;
            if (tout->edge_P) tout->edge_P[i] = edges[i].P;
            if (tout->edge_W) tout->edge_W[i] = edges[i].W;
            if (tout->edge_N) tout->edge_N[i] = edges[i].N;
        }
    }
    free(nodes);
    free(edges);
    free(path_e);
    free(path_n);
    free(pend_leaf);
    free(pend_depth);
    return chosen;
}

/* One search from a packed line.  root_* arrays hold up to 256 entries. */
KVO_API int kvo_mcts_search(const kvo_mcts_cfg *cfg, const uint64_t *line, uint64_t game_id, int ply,
                            const float *rep_node_val, const int32_t *rep_node_first, const float *rep_edge_P,
                            uint16_t *root_moves, uint32_t *root_N, float *root_W, float *root_P, int32_t *info4) {
    kvo_state s;
    kvo_unpack(line, &s);
    replay_t rep = { rep_node_val, rep_node_first, rep_edge_P };
    int n_root, nn, ne, ov;
    int mv = mcts_search(cfg, &s, game_id, ply, rep_node_val ? &rep : NULL, root_moves, root_N, root_W, root_P, &n_root,
                         &nn, &ne, &ov, NULL, NULL);
    info4[0] = n_root;
    info4[1] = nn;
    info4[2] = ne;
    info4[3] = ov;
    return mv;
}

/* kvo_mcts_search, and a copy of the tree it built (hash or replay mode): per node node_line [sims + 1][16],
 * node_i32 [sims + 1][4] = (terminal, first edge, edge count, N), node_val [sims + 1]; per edge [cfg->edge_cap] the
 * move word, child node, prior P, value sum W and visits N.  Nodes and edges are numbered in creation order, as on the
 * device.  Every output pointer may be NULL. */
KVO_API int kvo_mcts_search_tree(const kvo_mcts_cfg *cfg, const uint64_t *line, uint64_t game_id, int ply,
                                 const float *rep_node_val, const int32_t *rep_node_first, const float *rep_edge_P,
                                 uint16_t *root_moves, uint32_t *root_N, float *root_W, float *root_P, int32_t *info4,
                                 uint64_t *node_line, int32_t *node_i32, float *node_val, uint16_t *edge_mv,
                                 int32_t *edge_child, float *edge_P, float *edge_W, uint32_t *edge_N) {
    kvo_state s;
    kvo_unpack(line, &s);
    replay_t rep = { rep_node_val, rep_node_first, rep_edge_P };
    const tree_out_t tout = { node_line, node_i32, node_val, edge_mv, edge_child, edge_P, edge_W, edge_N };
    int n_root, nn, ne, ov;
    int mv = mcts_search(cfg, &s, game_id, ply, rep_node_val ? &rep : NULL, root_moves, root_N, root_W, root_P, &n_root,
                         &nn, &ne, &ov, NULL, &tout);
    info4[0] = n_root;
    info4[1] = nn;
    info4[2] = ne;
    info4[3] = ov;
    return mv;
}

/* test helper: the root noise eta[k] of priors_from_logits for a root with n legal moves (Gamma variates keyed by
 * ply * 256 + k, divided by their sequential sum) */
KVO_API void kvo_root_eta(float alpha, uint64_t seed, uint64_t game_id, int ply, int n, float *out) {
    float gs = 0.0f;
    for (int k = 0; k < n; k++) {
        out[k] = kvd_gamma_small(alpha, seed, game_id, (uint64_t)ply * 256 + (uint64_t)k);
        gs = gs + out[k];
    }
    for (int k = 0; k < n; k++) out[k] = out[k] / gs;
}

/* test helper: the Gamma(alpha) variates the reference-rule root noise draws for every policy index */
KVO_API void kvo_root_noise(float alpha, uint64_t seed, uint64_t game_id, int ply, float *out4096) {
    for (int i = 0; i < POLICY_N; i++)
        out4096[i] = kvd_gamma_small(alpha, seed, game_id, (uint64_t)ply * POLICY_N + (uint64_t)i);
}

/* test helper: the hash evaluator's logits for all 4096 policy indices and its white-perspective value */
KVO_API float kvo_hash_eval(const uint64_t *line, float *logits4096) {
    const uint64_t ph = pos_hash(line);
    for (int i = 0; i < POLICY_N; i++) logits4096[i] = hash_logit(ph, i);
    return hash_value(ph);
}

/* Whole self-play game (scripts/self_play.py:111-255 control flow; the move comes from the search, or from a script).
 * After every move the reference tests, in this order: isDraw() = only kings (:180) -> draw; resignation (:185-189:
 * move_count > resign_min_plies and the model's value of the position the move was chosen in < resign_thr ->
 * -1 if white is to move, else +1); max_moves (:196) -> draw even if the move mated (:209-211); and at the loop head
 * no legal move (:125) -> checkmate +-1 (:217-220) or stalemate 0 (:221-224).  The material branch (:229-238) is
 * unreachable through these exits and would yield 0.
 * script_moves / script_vals (nullable, script_n entries): per ply a move word to play instead of the search's choice
 * (matched on from/to; 0xFFFF = none) and the value the resign rule sees (NaN = the evaluator's root value).
 * out_moves[ply] = move word; out_lines[ply][16] = position the move was chosen in; returns the number of plies.
 * *result: +1 white won, -1 black won, 0 draw.  *out_flags: bit 1 = a scripted move was not legal. */
KVO_API int kvo_selfplay_game2(const kvo_mcts_cfg *cfg, const uint64_t *start_line, uint64_t game_id,
                               const uint16_t *script_moves, const float *script_vals, int script_n, uint16_t *out_moves,
                               uint64_t *out_lines, int32_t *result, int32_t *out_flags) {
    kvo_state s;
    kvo_unpack(start_line, &s);
    uint16_t rm[256];
    uint32_t rn[256];
    float rw[256], rp[256];
    int ply = 0;
    *result = 0;
    if (out_flags) *out_flags = 0;
    for (;;) {
        kvo_state probe = s;
        movelist ml;
        int f;
        int n = valid_moves(&probe, &ml, &f);
        s = probe;   /* getValidMoves may rewrite the state */
        if (n == 0) {                                    /* :125, then :217-224 */
            if (f & RF_CHECKMATE) *result = s.white_to_move ? -1 : 1;
            break;
        }
        if (ply == 0 && (f & RF_ONLY_KINGS)) break;      /* a start position without pieces: nothing to search */
        int n_root, nn, ne, ov;
        float vroot = 0.0f;
        int mv = mcts_search(cfg, &s, game_id, ply, NULL, rm, rn, rw, rp, &n_root, &nn, &ne, &ov, &vroot, NULL);
        if (ply < script_n) {
            if (script_vals && script_vals[ply] == script_vals[ply]) vroot = script_vals[ply];
            if (script_moves && script_moves[ply] != 0xFFFF) {
                int found = -1;
                for (int k = 0; k < n_root && found < 0; k++)
                    if ((rm[k] & 0xFFF) == (script_moves[ply] & 0xFFF)) found = k;
                if (found < 0) {
                    if (out_flags) *out_flags |= 2;
                    break;
                }
                mv = rm[found];
            }
        }
        kvo_pack(&s, out_lines + 16 * (size_t)ply);
        out_moves[ply] = (uint16_t)mv;
        make_move(&s, mv & 63, (mv >> 6) & 63, (mv >> 12) & 7, T_Q);
        ply++;
        if (only_kings(&s)) break;                                                      /* :180 */
        if (cfg->resign_min_plies >= 0 && ply > cfg->resign_min_plies && vroot < cfg->resign_thr) {
            *result = s.white_to_move ? -1 : 1;                                         /* :185-189 */
            break;
        }
        if (ply >= cfg->max_plies) break;                                               /* :196 */
    }
    return ply;
}

KVO_API int kvo_selfplay_game(const kvo_mcts_cfg *cfg, const uint64_t *start_line, uint64_t game_id, uint16_t *out_moves,
                              uint64_t *out_lines, int32_t *result) {
    return kvo_selfplay_game2(cfg, start_line, game_id, NULL, NULL, 0, out_moves, out_lines, result, NULL);
}


/* ==========================================================================================================
 * Step-wise form of the sequential search (K = 1, legal-move priors) with an EXTERNAL evaluator: select a leaf, hand
 * its position out, take the evaluator's logits and value back.  bench.py's CPU arm drives many games in lock step so
 * that the fp32 network (torch CPU kernels) sees a batch, the way the device engine batches its leaves.  Same
 * arithmetic as mcts_search / kvo_selfplay_game2 (tests/test_oracle_step_api.py feeds it the hash evaluator's logits
 * and gets the same games bit for bit).
 * ========================================================================================================== */
typedef struct {
    kvo_mcts_cfg cfg;
    kvo_state st;            /* current position of the game */
    uint64_t game_id;
    onode *nodes;
    oedge *edges;
    int *path_e, *path_n;
    int n_nodes, n_edges, sims_done, ply, done, result, overflow;
    int pend_leaf, pend_depth;
    uint16_t *rec_moves;     /* moves played so far [max_plies] */
} kvo_tree;

KVO_API void *kvo_tree_new(const kvo_mcts_cfg *cfg, const uint64_t *start_line, uint64_t game_id) {
    kvo_tree *t = (kvo_tree *)calloc(1, sizeof(kvo_tree));
    t->cfg = *cfg;
    kvo_unpack(start_line, &t->st);
    t->game_id = game_id;
    t->nodes = (onode *)calloc((size_t)cfg->sims + 1, sizeof(onode));
    t->edges = (oedge *)calloc((size_t)cfg->edge_cap, sizeof(oedge));
    t->path_e = (int *)malloc(sizeof(int) * ((size_t)cfg->sims + 2));
    t->path_n = (int *)malloc(sizeof(int) * ((size_t)cfg->sims + 2));
    t->rec_moves = (uint16_t *)calloc((size_t)(cfg->max_plies > 0 ? cfg->max_plies : 1), sizeof(uint16_t));
    t->pend_leaf = -1;
    return t;
}

KVO_API void kvo_tree_free(void *tp) {
    kvo_tree *t = (kvo_tree *)tp;
    if (!t) return;
    free(t->nodes); free(t->edges); free(t->path_e); free(t->path_n); free(t->rec_moves);
    free(t);
}

/* Selections until one needs the evaluator.  Returns 1: a leaf is waiting (its line, the policy indices of its legal
 * moves in edge order and their count are written); 0: the move's simulations are complete, call kvo_tree_finish_move;
 * -1: the game is over. */
KVO_API int kvo_tree_select(void *tp, uint64_t *leaf_line16, int32_t *legal_idx256, int32_t *n_legal) {
    kvo_tree *t = (kvo_tree *)tp;
    const kvo_mcts_cfg *cfg = &t->cfg;
    if (t->done) return -1;
    while (t->sims_done < cfg->sims) {
        int depth = 0, node = 0, leaf = -1;
        float v = 0.0f;
        kvo_state child_st;
        if (t->n_nodes == 0) {
            child_st = t->st;
            leaf = 0;
        } else {
            for (;;) {
                onode *nd = &t->nodes[node];
                if (nd->term) {
                    v = nd->val;
                    nd->N++;
                    break;
                }
                const float sq = KVD_SQRTF((float)nd->N);
                int best = 0;
                float bs = 0.0f;
                for (int k = 0; k < nd->n_edges; k++) {
                    const oedge *e = &t->edges[nd->first_edge + k];
                    float sc = kvd_puct(e->W, e->N, e->P, sq, cfg->c_puct);
                    if (k == 0 || sc > bs) { bs = sc; best = k; }
                }
                const int ei = nd->first_edge + best;
                t->path_n[depth] = node;
                t->path_e[depth] = ei;
                depth++;
                t->edges[ei].VL++;      /* backup_path turns the virtual visit into the real one */
                nd->VL++;
                if (t->edges[ei].child < 0) {
                    child_st = nd->st;
                    make_move(&child_st, t->edges[ei].mv & 63, (t->edges[ei].mv >> 6) & 63, (t->edges[ei].mv >> 12) & 7, T_Q);
                    leaf = t->n_nodes;
                    t->edges[ei].child = leaf;
                    break;
                }
                node = t->edges[ei].child;
            }
        }
        if (leaf >= 0) {
            onode *nd = &t->nodes[leaf];
            movelist ml;
            int f;
            int n = valid_moves(&child_st, &ml, &f);
            if (n > 256) n = 256;
            memset(nd, 0, sizeof(*nd));
            nd->st = child_st;
            nd->N = 1;
            nd->first_edge = -1;
            t->n_nodes++;
            if (n == 0) {
                nd->term = 1;
                nd->val = (f & RF_CHECKMATE) ? -1.0f : 0.0f;
            } else if (f & RF_ONLY_KINGS) {
                nd->term = 1;
            } else if (t->n_edges + n > cfg->edge_cap) {
                nd->term = 1;
                t->overflow = 1;
            } else {
                nd->first_edge = t->n_edges;
                nd->n_edges = n;
                oedge *e = &t->edges[t->n_edges];
                t->n_edges += n;
                for (int k = 0; k < n; k++) {
                    e[k].mv = pack_move(&ml.m[k]);
                    e[k].N = 0; e[k].VL = 0; e[k].W = 0.0f; e[k].P = 0.0f; e[k].child = -1;
                    legal_idx256[k] = kvo_move_index(e[k].mv);
                }
                *n_legal = n;
                kvo_pack(&nd->st, leaf_line16);
                t->pend_leaf = leaf;
                t->pend_depth = depth;
                return 1;
            }
            v = nd->val;
        }
        backup_path(t->nodes, t->edges, t->path_n, t->path_e, depth, v);
        t->sims_done++;
    }
    return 0;
}

/* The evaluator's answer for the waiting leaf: logits of its legal moves (edge order) and the white-perspective value */
KVO_API void kvo_tree_expand(void *tp, const float *legal_logits, float v_white) {
    kvo_tree *t = (kvo_tree *)tp;
    if (t->pend_leaf < 0) return;
    onode *nd = &t->nodes[t->pend_leaf];
    oedge *e = &t->edges[nd->first_edge];
    float mx = 0.0f;
    for (int k = 0; k < nd->n_edges; k++) {
        e[k].P = legal_logits[k];
        if (k == 0 || e[k].P > mx) mx = e[k].P;
    }
    priors_from_logits(&t->cfg, e, nd->n_edges, mx, t->pend_leaf == 0, t->game_id, t->ply);
    nd->val = nd->st.white_to_move ? v_white : -v_white;
    backup_path(t->nodes, t->edges, t->path_n, t->path_e, t->pend_depth, nd->val);
    t->sims_done++;
    t->pend_leaf = -1;
}

/* After the move's simulations: choose, play, apply the game-loop rules (kvo_selfplay_game2's).  Returns 1 while the
 * game goes on, 0 when it ended. */
KVO_API int kvo_tree_finish_move(void *tp) {
    kvo_tree *t = (kvo_tree *)tp;
    const kvo_mcts_cfg *cfg = &t->cfg;
    if (t->done) return 0;
    if (t->n_nodes == 0 || t->nodes[0].term) {
        t->done = 1;
        t->result = (t->n_nodes && t->nodes[0].val < 0.0f) ? (t->st.white_to_move ? -1 : 1) : 0;
        return 0;
    }
    const onode *root = &t->nodes[0];
    const oedge *e = &t->edges[root->first_edge];
    uint64_t total = 0;
    for (int k = 0; k < root->n_edges; k++) total += e[k].N;
    const float vroot = root->st.white_to_move ? root->val : -root->val;
    const int mv = e[choose_move(cfg, e, root->n_edges, total, t->game_id, t->ply)].mv;
    t->st = root->st;          /* carries a getValidMoves rewrite, as the reference's state would */
    if (t->ply < cfg->max_plies) t->rec_moves[t->ply] = (uint16_t)mv;
    make_move(&t->st, mv & 63, (mv >> 6) & 63, (mv >> 12) & 7, T_Q);
    t->ply++;
    t->n_nodes = t->n_edges = t->sims_done = 0;
    if (only_kings(&t->st)) {
        t->done = 1;
    } else if (cfg->resign_min_plies >= 0 && t->ply > cfg->resign_min_plies && vroot < cfg->resign_thr) {
        t->done = 1;
        t->result = t->st.white_to_move ? -1 : 1;
    } else if (t->ply >= cfg->max_plies) {
        t->done = 1;
    } else {
        kvo_state probe = t->st;
        movelist ml;
        int f;
        if (valid_moves(&probe, &ml, &f) == 0) {
            t->done = 1;
            t->result = (f & RF_CHECKMATE) ? (t->st.white_to_move ? -1 : 1) : 0;
        }
    }
    return !t->done;
}

/* info5: ply, done, result, simulations done in the current move, overflow; moves (nullable): the plies played */
KVO_API void kvo_tree_info(void *tp, int32_t *info5, uint16_t *moves) {
    kvo_tree *t = (kvo_tree *)tp;
    info5[0] = t->ply; info5[1] = t->done; info5[2] = t->result; info5[3] = t->sims_done; info5[4] = t->overflow;
    if (moves) memcpy(moves, t->rec_moves, sizeof(uint16_t) * (size_t)(t->ply < t->cfg.max_plies ? t->ply : t->cfg.max_plies));
}
