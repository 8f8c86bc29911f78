"""Positions for the endgame-solver tests, drawn from the oracle's engine-RNG playouts (no device needed)."""
import numpy as np


def empties(own: int, opp: int, n: int) -> int:
    return n * n - bin(int(own) | int(opp)).count("1")


def playout_positions(O, n, count, max_empties, seed, min_empties=0):
    """`count` positions (own, opp, player) with min_empties..max_empties empties from random playouts of the oracle O:
    positions along each game (side to move = own), the same position with the other side to move (which includes
    positions whose mover must pass), and finished positions."""
    rng = np.random.default_rng(seed)
    out, g = [], 0
    while len(out) < count:
        full = O.playout(n, seed, g)
        k = len(full["moves"])
        g += 1
        for back in sorted(set(int(b) for b in rng.integers(0, max(1, k), 3))):
            st = O.playout(n, seed, g - 1, max_moves=k - back) if back else full
            own, opp = (st["black"], st["white"]) if st["player"] == 0 else (st["white"], st["black"])
            if min_empties <= empties(own, opp, n) <= max_empties:
                out.append((own, opp, st["player"]))
                out.append((opp, own, 1 - st["player"]))
    return out[:count]


def kinds(O, positions, n):
    """Counts of finished positions, positions whose mover must pass, and positions with a move after which the
    opponent must pass (a pass inside the solved tree)."""
    fin = root_pass = inner_pass = 0
    for own, opp, _ in positions:
        b = O.bits_to_board(int(own), int(opp), n)   # channel 0 = the side to move
        mine, theirs = O.valid_actions(b, 0), O.valid_actions(b, 1)
        if not mine:
            fin += not theirs
            root_pass += bool(theirs)
            continue
        for r, c in mine:
            child = O.flip_board(b, 0, r, c)
            if not O.valid_actions(child, 1) and O.valid_actions(child, 0):
                inner_pass += 1
                break
    return dict(finished=fin, root_pass=root_pass, inner_pass=inner_pass)


def oracle_margins(O, positions, n, per_move=False):
    """Oracle solver margins (mover = own = channel 0), and per-move rows [64] (SOLVE_NONE off the legal moves)."""
    margin = np.array([O.solve_margin(O.bits_to_board(int(o), int(p), n), 0) for o, p, _ in positions], dtype=np.int64)
    if not per_move:
        return margin
    rows = np.full((len(positions), 64), -128, dtype=np.int64)
    for i, (o, p, _) in enumerate(positions):
        for sq, v in O.solve_move_margins(O.bits_to_board(int(o), int(p), n), 0).items():
            rows[i, sq] = v
    return margin, rows
