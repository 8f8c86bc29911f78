"""Rules side of the drop-in: the reference's ``Othello`` module API (Othello/__init__.py) with every
rule evaluated by the CUDA bitboard kernels (K1/K2) through the C-ABI.

Same names, argument meaning and error behaviour as the reference so that training.py / agents.py /
othelo_mcts.py keep working when they import ``OthelloGame`` from here.  Boards are the reference's
``(N,N,2)`` bool arrays (channel 0 = BLACK, 1 = WHITE); each call converts to two uint64 bitboards (vectorised)
and launches a kernel for ONE position — the interface the reference's per-game callers expect.  Many positions at once
go through engine.legal_moves / apply_moves / score (arena.pit) or the batched engine (selfplay.py).  The reference's
ray generators (get_direction_squares / get_all_directions_squares, :186-198) have no counterpart: rays are shift masks
inside the kernels (csrc/oz_bitboard.cuh).

Deliberate deviations are listed in INTEGRATION.md (e.g. ``is_square_free`` works here; the reference's
version raises NameError, Othello/__init__.py:88-98).

``OthelloGame`` plays the reference's rules, including its flip rule (a move also flips opponent discs beyond the
bracketing own disc).  ``StandardOthelloGame`` is the same class with standard Othello flipping; the class attribute
``rules`` selects the rule set of ``play``, ``get_action_flip_squares``, ``flip_board_squares`` and ``getNextState``.
Both count a draw as a BLACK win, like the reference.  The class attribute ``scoring = "standard"`` scores it as a draw
instead: ``get_board_winning_player`` / ``get_winning_player`` return ``(None, points)`` and ``getGameEnded`` returns
1e-4 (alpha-zero-general's small non-zero value for a draw).  ``game_class(rules, scoring)`` returns the class for any
combination.
"""
from __future__ import annotations

from enum import Enum, auto

import numpy as np

from . import engine as _e
from ._lib import MOVE_FINISHED, MOVE_SWAPPED, board_arg


class BoardView(Enum):
    ONE_CHANNEL = auto()
    TWO_CHANNELS = auto()


class OthelloPlayer(Enum):
    """Othello/__init__.py:12-18."""
    BLACK = 1
    WHITE = -1

    @property
    def opponent(self):
        return OthelloPlayer(-self.value)


_SQUARE_BIT = (np.uint64(1) << (np.arange(8, dtype=np.uint64)[:, None] * np.uint64(8) + np.arange(8, dtype=np.uint64)[None, :]))


def _bits(board) -> tuple[int, int]:
    """(N,N,2) board -> (channel 0 bits, channel 1 bits), bit r*8+c; one masked sum per channel, no Python loop."""
    b = np.asarray(board).astype(bool)
    n = b.shape[0]
    w = _SQUARE_BIT[:n, :n]
    return int(w[b[..., 0]].sum(dtype=np.uint64)), int(w[b[..., 1]].sum(dtype=np.uint64))


def _planes(bits: int, n: int) -> np.ndarray:
    """uint64 -> (N,N) bool plane (byte r of the little-endian word = row r)."""
    rows = np.frombuffer(int(bits).to_bytes(8, "little"), dtype=np.uint8)
    return np.unpackbits(rows[:, None], axis=1, bitorder="little")[:n, :n].astype(bool)


def _mask_to_squares(mask: int, n: int):
    rr, cc = np.nonzero(_planes(mask, n))           # row-major, like np.argwhere in the reference (:200-210)
    return list(zip(rr.tolist(), cc.tolist()))


class OthelloGame:
    PLAYER_CHANNELS = {OthelloPlayer.BLACK: 0, OthelloPlayer.WHITE: 1}
    device = 0  # CUDA ordinal used by the static rule calls
    rules = "reference"  # flip rule of play / get_action_flip_squares / flip_board_squares / getNextState
    scoring = "reference"  # "standard": equal counts are a draw in get_board_winning_player / getGameEnded

    def __init__(self, board_size=8, initial_board=None, current_player=OthelloPlayer.BLACK):
        """Othello/__init__.py:29-59: same arguments, same assertions; a supplied board is adopted (not copied)."""
        assert board_size % 2 == 0, 'Board size must be even'
        if initial_board is None:
            initial_board = self.initial_board(board_size)
            finished = False
        else:
            assert initial_board.shape == (board_size, board_size, 2), \
                f'Expecting initial board shape ({board_size}, {board_size}, 2)'
            finished = OthelloGame.has_board_finished(initial_board)
        self._board, self._board_size, self._round = initial_board, board_size, 1
        self.current_player = current_player
        self._has_finished = finished
        self._one_channel_cache = (None, None)   # (round it was built in, array)

    # ---- instance API (Othello/__init__.py:61-175) ----------------------------------------------
    @property
    def board_size(self):
        return self._board_size

    @property
    def round(self):
        return self._round

    def board(self, view=BoardView.ONE_CHANNEL):
        """:77-86 - TWO_CHANNELS hands out the LIVE array (callers alias it, SURVEY 0.8); ONE_CHANNEL is rebuilt once
        per round."""
        if not isinstance(view, BoardView):
            raise TypeError('Expecting BoardView type')
        if view is BoardView.TWO_CHANNELS:
            return self._board
        if self._one_channel_cache[0] != self._round:
            self._one_channel_cache = (self._round, OthelloGame.convert_to_one_channel_board(self._board))
        return self._one_channel_cache[1]

    def is_square_free(self, row, col):
        return OthelloGame.is_board_square_free(self._board, row, col)

    def is_valid_action(self, row, col):
        return OthelloGame.is_valid_player_action(self._board, self.current_player, row, col)

    def get_valid_actions(self):
        return OthelloGame.get_player_valid_actions(self._board, self.current_player)

    def get_free_squares(self):
        return OthelloGame.get_board_free_squares(self._board)

    def has_finished(self):
        return self._has_finished

    def play(self, row, col):
        """Othello/__init__.py:136-159 — one K2 launch does the flips and the pass/terminal test."""
        assert not self._has_finished, 'Game has ended'
        n = self._board_size
        black, white = _bits(self._board)
        own, opp = (black, white) if self.current_player is OthelloPlayer.BLACK else (white, black)
        o2, p2, fl, _ = _e.apply_moves([own], [opp], [int(row) * 8 + int(col)], n, self.device, rules=self.rules)
        fl = int(fl[0])
        if fl & 0x80000000:
            # the reference does not validate: it places the disc and flips nothing (:237-247)
            o2, p2, fl = self._play_unchecked(own, opp, int(row) * 8 + int(col))
        swapped = bool(fl & MOVE_SWAPPED)
        mover_bits, other_bits = (int(p2[0]), int(o2[0])) if swapped else (int(o2[0]), int(p2[0]))
        nb, nw = (mover_bits, other_bits) if self.current_player is OthelloPlayer.BLACK else (other_bits, mover_bits)
        self._write_bits(nb, nw)
        self._round += 1
        if fl & MOVE_FINISHED:
            self.current_player = self.current_player.opponent  # :147 — switched, never switched back
            self._has_finished = True
        elif swapped:
            self.current_player = self.current_player.opponent

    def _play_unchecked(self, own, opp, sq):
        own |= 1 << sq
        opp &= ~(1 << sq)
        n = self._board_size
        lo = int(_e.legal_moves([opp], [own], n, self.device)[0])
        if lo:
            return np.array([opp], dtype=np.uint64), np.array([own], dtype=np.uint64), MOVE_SWAPPED
        lm = int(_e.legal_moves([own], [opp], n, self.device)[0])
        return np.array([own], dtype=np.uint64), np.array([opp], dtype=np.uint64), (2 if lm else MOVE_FINISHED)

    def _write_bits(self, black, white):
        n = self._board_size
        self._board[..., 0] = _planes(black, n)     # in place: the array is shared with whoever holds board(TWO_CHANNELS)
        self._board[..., 1] = _planes(white, n)

    def get_players_points(self):
        return OthelloGame.get_board_players_points(self._board)

    def get_winning_player(self):
        return self.get_board_winning_player(self._board)

    # ---- static array API (Othello/__init__.py:177-274) -----------------------------------------
    @staticmethod
    def initial_board(board_size):
        """:177-184 - WHITE on the main diagonal of the centre 2x2, BLACK on the other two squares."""
        assert board_size % 2 == 0, 'Board size must be even'
        board = np.zeros((board_size, board_size, 2), dtype=bool)
        lo, hi = board_size // 2 - 1, board_size // 2
        board[[lo, hi], [lo, hi], 1] = True
        board[[lo, hi], [hi, lo], 0] = True
        return board

    @staticmethod
    def get_board_free_squares(board):
        return np.argwhere(~np.asarray(board, dtype=bool).any(axis=2))   # row-major, like the reference's argwhere

    @staticmethod
    def is_board_square_free(board, row, col):
        return np.logical_not(np.asarray(board[row, col], dtype=bool).any())

    @staticmethod
    def _own_opp(board, player):
        if not isinstance(player, OthelloPlayer):
            raise TypeError('Expecting OthelloPlayer type')
        black, white = _bits(board)
        return (black, white) if player is OthelloPlayer.BLACK else (white, black)

    @staticmethod
    def legal_mask(board, player) -> int:
        own, opp = OthelloGame._own_opp(board, player)
        return int(_e.legal_moves([own], [opp], np.asarray(board).shape[0], OthelloGame.device)[0])

    @staticmethod
    def get_player_valid_actions(board, player):
        """Generator of [row, col] arrays in row-major order (:208-210)."""
        n = np.asarray(board).shape[0]
        mask = OthelloGame.legal_mask(board, player)
        return (np.array([r, c]) for r, c in _mask_to_squares(mask, n))

    @staticmethod
    def is_valid_player_action(board, player, row, col):
        return bool((OthelloGame.legal_mask(board, player) >> (int(row) * 8 + int(col))) & 1)

    @classmethod
    def get_action_flip_squares(cls, board, player, row, col):
        """The SET of flipped squares in row-major order (the reference's generator also yields duplicates,
        :216-235; every consumer only uses membership), under ``cls.rules``."""
        n = np.asarray(board).shape[0]
        own, opp = OthelloGame._own_opp(board, player)
        sq = int(row) * 8 + int(col)
        if (own | opp) >> sq & 1:
            return iter(())
        o2, p2, fl, _ = _e.apply_moves([own], [opp], [sq], n, cls.device, rules=cls.rules)
        if int(fl[0]) & 0x80000000:
            return iter(())
        mover = int(p2[0]) if int(fl[0]) & MOVE_SWAPPED else int(o2[0])
        flipped = mover & ~own & ~(1 << sq)
        return iter(_mask_to_squares(flipped, n))

    @classmethod
    def flip_board_squares(cls, board, player, row, col):
        """:237-247, in place: the flipped squares and the played square go to `player`'s channel."""
        mine = cls.PLAYER_CHANNELS[player]
        squares = list(cls.get_action_flip_squares(board, player, row, col)) + [(row, col)]
        rr, cc = zip(*squares)
        board[rr, cc, mine] = True
        board[rr, cc, 1 - mine] = False

    @staticmethod
    def has_board_finished(board):
        return not OthelloGame.has_player_actions_on_board(board, OthelloPlayer.BLACK) and \
            not OthelloGame.has_player_actions_on_board(board, OthelloPlayer.WHITE)

    @classmethod
    def get_board_winning_player(cls, board):
        """-> (winning OthelloPlayer, its points).  A draw goes to BLACK (dict order, :254-256), or under standard scoring
        is (None, points)."""
        points = OthelloGame.get_board_players_points(board)
        top = max(points.values())
        if cls.scoring == "standard" and points[OthelloPlayer.BLACK] == points[OthelloPlayer.WHITE]:
            return None, top
        return next((player, count) for player, count in points.items() if count == top)   # draw -> BLACK (dict order)

    @staticmethod
    def get_board_players_points(board):
        black, white = _bits(board)
        cb, cw = _e.score([black], [white], OthelloGame.device)
        return {OthelloPlayer.BLACK: int(cb[0]), OthelloPlayer.WHITE: int(cw[0])}

    @staticmethod
    def has_player_actions_on_board(board, player):
        return OthelloGame.legal_mask(board, player) != 0

    @staticmethod
    def convert_to_one_channel_board(board):
        """:266-270 - +1 where BLACK, -1 where WHITE (the players' enum values), 0 elsewhere."""
        b = np.asarray(board)
        return b[..., 0] * OthelloPlayer.BLACK.value + b[..., 1] * OthelloPlayer.WHITE.value

    @staticmethod
    def invert_board(board):
        return board[..., ::-1]   # a view with the two channels swapped

    # ---- alpha-zero-general style aliases named in BASELINE.json (SURVEY Appendix D) --------------
    getInitBoard = initial_board

    @staticmethod
    def getValidMoves(board, player):
        n = np.asarray(board).shape[0]
        mask = OthelloGame.legal_mask(board, player)
        out = np.zeros((n, n), dtype=np.float64)
        for r, c in _mask_to_squares(mask, n):
            out[r, c] = 1
        return out

    @classmethod
    def getNextState(cls, board, player, action):
        """-> (next_board, next_player) with OthelloGame.play's pass handling, under ``cls.rules``."""
        b = np.array(board, copy=True)
        g = cls(b.shape[0], initial_board=b, current_player=player)
        g._has_finished = False
        g.play(*action)
        return g.board(BoardView.TWO_CHANNELS), g.current_player

    @classmethod
    def getGameEnded(cls, board):
        """0 if not ended, else the winner's OthelloPlayer.value (draw -> BLACK; under standard scoring a draw is 1e-4)."""
        if not OthelloGame.has_board_finished(board):
            return 0
        winner = cls.get_board_winning_player(board)[0]
        return 1e-4 if winner is None else winner.value

    @staticmethod
    def getCanonicalForm(board, player):
        return OthelloGame.invert_board(board) if player is OthelloPlayer.WHITE else board


class StandardOthelloGame(OthelloGame):
    """OthelloGame with standard Othello flipping: a run of opponent discs flips only up to the first own disc beyond
    it.  Legal moves, passes, the end of the game and the scoring (a draw counts as a BLACK win) are unchanged."""
    rules = "standard"


_game_classes = {("reference", "reference"): OthelloGame, ("standard", "reference"): StandardOthelloGame}


def game_class(rules: str = "reference", scoring: str = "reference") -> type:
    """The game class for a rule set and a scoring: ``OthelloGame`` or ``StandardOthelloGame`` under reference scoring,
    otherwise a subclass of one of them with ``scoring = "standard"`` (made once, then cached).  Unknown values raise
    ValueError."""
    board_arg(8, rules, scoring)
    key = (rules, scoring)
    if key not in _game_classes:
        base = _game_classes[(rules, "reference")]
        _game_classes[key] = type(base.__name__ + "StandardScoring", (base,), {
            "scoring": scoring, "__module__": __name__,
            "__doc__": f"{base.__name__} with standard scoring: a finished game with equal disc counts is a draw."})
    return _game_classes[key]
