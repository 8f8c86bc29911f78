"""Episode side of the drop-in: ``training.execute_episode`` (training.py:26-72) and a ``workers.Worker``
(workers.py:24-79) that plays all of its episodes as ONE batch on the GPU.

    examples = execute_episode(board_size, neural_network, degree_exploration,
                               num_simulations, policy_temperature, e_greedy)

returns the reference's list of ``(board (N,N,2) bool, one-hot policy (N,N) float64, z)`` with the 8
symmetries of training.py:13-23 in the reference's order.  Differences, all documented in INTEGRATION.md:
boards are true per-move snapshots unless ``reference_aliasing=True`` (the reference aliases the live board,
SURVEY §0.8); with e_greedy < 1 the random moves come from the engine's counter RNG, not CPython's.
Every entry point takes ``rules="reference"`` (the reference's flip rule) or ``rules="standard"`` (standard Othello),
and ``scoring="reference"`` (a draw counts as a BLACK win) or ``scoring="standard"`` (a draw is a draw: winner code 2,
z = 0 for every example of the game).
"""
from __future__ import annotations

import logging
import os
import threading
import uuid

import numpy as np

from . import engine as _e
from ._lib import WINNER_DRAW
from .mcts import HashPriorNet
from .net import B200NNet


def training_example_symmetries(board, policy):
    """The 8 symmetric copies in the order of training.py:13-23: for 1..4 quarter turns, the mirrored copy first."""
    pairs = []
    for quarter_turns in (1, 2, 3, 4):
        rb, rp = np.rot90(board, quarter_turns), np.rot90(policy, quarter_turns)
        pairs.append((np.fliplr(rb), np.fliplr(rp)))
        pairs.append((rb, rp))
    return pairs


getSymmetries = training_example_symmetries  # alpha-zero-general name (SURVEY Appendix D)


def default_nodes_per_game(board_size: int, num_simulations: int) -> int:
    # the reference never prunes: <= one new node per simulation for every move of the episode
    return num_simulations * (board_size * board_size - 4) + 64


class SelfPlay:
    """A pool of concurrent self-play games on one GPU (one warp per game)."""

    def __init__(self, board_size: int, neural_network, degree_exploration: float = 1.0, max_games: int = 4096,
                 num_simulations: int = 100, device: int = 0, seed: int = 0, log_visits: bool = False,
                 eval_cache_log2: int = 22, rules: str = "reference", scoring: str = "reference"):
        self.board_size = board_size
        self.num_simulations = num_simulations
        if isinstance(neural_network, HashPriorNet):
            mode = _e.PRIOR_HASH
        elif isinstance(neural_network, B200NNet):
            mode = _e.PRIOR_NET
        else:
            raise TypeError("device self-play needs a B200NNet or HashPriorNet; for any other net object use "
                            "othellozero_b200.mcts.OthelloMCTS (host-evaluated priors)")
        self.engine = _e.Engine(board_size, max_games=max_games,
                                nodes_per_game=default_nodes_per_game(board_size, num_simulations), prior_mode=mode,
                                c_puct=float(degree_exploration), seed=seed, device=device, log_visits=log_visits,
                                # identical positions reached by different games are evaluated once (results unchanged:
                                # tests/test_gpu_net.py::test_eval_cache_is_results_preserving); 272 B per entry
                                eval_cache_log2=eval_cache_log2 if mode == _e.PRIOR_NET else 0, rules=rules,
                                scoring=scoring)
        if mode == _e.PRIOR_NET:
            self.engine.load_weights(neural_network.blob, neural_network.channels, neural_network.precision)

    def set_weights(self, blob, channels):
        self.engine.load_weights(blob, channels, self.engine.precision)

    def play(self, n_games: int, policy_temperature: float = 1.0, e_greedy: float = 1.0, game_ids=None,
             black=None, white=None, player=None, max_moves: int = -1) -> dict:
        self.engine.selfplay_begin(n_games, self.num_simulations, policy_temperature, e_greedy, max_moves, black, white,
                                   player, game_ids)
        self.engine.selfplay_run(-1)
        return self.engine.selfplay_records()

    def close(self):
        self.engine.close()


def records_to_examples(rec: dict, game: int, board_size: int, reference_aliasing: bool = False):
    """One game's records -> the reference's example list (training.py:58-72): per move the 8 symmetries of
    (board (N,N,2) bool, one-hot policy (N,N) float64) in the order of training.py:13-23, with z = +1 iff the mover won
    (z = 0 for every example of a drawn game, winner code 2, which only standard scoring records).

    reference_aliasing=True reproduces the reference's stream byte for byte: its examples hold VIEWS of the live board
    (training.py:63 appends np.rot90 / np.fliplr views of game.board()), so once the episode is over every example shows
    the final position (SURVEY 0.8).  The final position is entry n_moves of the record row (include/oz_b200.h)."""
    n = board_size
    k = int(rec["n_moves"][game])
    winner = int(rec["winner"][game])
    examples = []
    if reference_aliasing:
        final_board = bits_to_boards(rec["black"][game][k:k + 1], rec["white"][game][k:k + 1], n)[0]
    else:
        boards = bits_to_boards(rec["black"][game][:k], rec["white"][game][:k], n)
    for p in range(k):
        board = final_board if reference_aliasing else boards[p]
        a = int(rec["action"][game][p])
        policy = np.zeros((n, n))
        policy[a >> 3][a & 7] = 1
        z = 0 if winner == WINNER_DRAW else (1 if winner == int(rec["player"][game][p]) else -1)
        for b, pol in training_example_symmetries(board, policy):
            examples.append((b, pol, z))
    return examples


def bits_to_boards(black, white, board_size: int) -> np.ndarray:
    """uint64 bitboards [P] -> (P, N, N, 2) bool in the reference's layout (channel 0 BLACK, bit r*8+c), vectorised."""
    def planes(x):
        b = np.ascontiguousarray(x, dtype="<u8").view(np.uint8).reshape(-1, 8)          # byte r = row r
        return np.unpackbits(b, axis=1, bitorder="little").reshape(-1, 8, 8)[:, :board_size, :board_size]
    return np.stack([planes(black), planes(white)], axis=-1).astype(bool)


def expand_symmetries(black, white, action, board_size: int):
    """Positions [P] (bitboards + action square bit) -> (boards (P,8,N,N,2) bool, one-hot policies (P,8,N,N) float64):
    the 8 symmetric copies of training.py:13-23, in its order, for every position at once."""
    n = board_size
    boards = bits_to_boards(black, white, n)
    action = np.asarray(action).astype(np.int64)
    P = boards.shape[0]
    b8 = np.empty((P, 8, n, n, 2), dtype=bool)
    p8 = np.zeros((P, 8, n, n))                  # one-hot policies: set the image of the action square under each symmetry
    rows, ar, ac = np.arange(P), action >> 3, action & 7
    s = 0
    for quarter_turns in (1, 2, 3, 4):
        rb = np.rot90(boards, k=quarter_turns, axes=(1, 2))
        ar, ac = n - 1 - ac, ar                                                          # np.rot90: out[i, j] = in[j, n-1-i]
        for mirrored in (True, False):                                                   # the mirrored copy comes first
            b8[:, s] = rb[:, :, ::-1] if mirrored else rb                                # np.fliplr of one (N,N,.) board
            p8[rows, s, ar, (n - 1 - ac) if mirrored else ac] = 1
            s += 1
    return b8, p8


def records_to_examples_batch(rec: dict, board_size: int, games=None, winners=None):
    """All games' records -> per-game example lists (training.py:58-72 + the 8 symmetries of :13-23), built with array
    operations over every (game, ply) at once: ~40x faster than calling records_to_examples per game (45 s -> ~1 s per
    4096 8x8 games).  The tuples hold views into three big arrays; order and values equal records_to_examples'.
    winners: optional per-position winner codes [G, 64] (solve_record_winners) in place of each game's winner."""
    n = board_size
    games = range(len(rec["n_moves"])) if games is None else list(games)
    nm = np.asarray([int(rec["n_moves"][g]) for g in games], dtype=np.int64)
    gsel = np.repeat(np.asarray(list(games), dtype=np.int64), nm)                        # game of every (game, ply) row
    psel = np.concatenate([np.arange(k) for k in nm]) if len(nm) else np.zeros(0, dtype=np.int64)
    P = int(gsel.size)
    b8, p8 = expand_symmetries(np.asarray(rec["black"])[gsel, psel], np.asarray(rec["white"])[gsel, psel],
                               np.asarray(rec["action"])[gsel, psel], n)
    w = np.asarray(rec["winner"])[gsel] if winners is None else np.asarray(winners)[gsel, psel]
    z = np.where(w == WINNER_DRAW, 0, np.where(w == np.asarray(rec["player"])[gsel, psel], 1, -1))
    # one (board view, policy view, z) tuple per example, made by C-level iteration over the leading axis
    flat = list(zip(b8.reshape(P * 8, n, n, 2), p8.reshape(P * 8, n, n), np.repeat(np.asarray(z, dtype=np.int64), 8).tolist()))
    out, row = [], 0
    for k in nm:
        out.append(flat[row:row + 8 * int(k)])
        row += 8 * int(k)
    return out


def solvable_positions(rec: dict, board_size: int, empties: int) -> np.ndarray:
    """[G, 64] bool: the recorded positions (before their move) with at most `empties` empty squares."""
    both = np.asarray(rec["black"], dtype=np.uint64) | np.asarray(rec["white"], dtype=np.uint64)
    discs = np.unpackbits(both.view(np.uint8).reshape(both.shape + (8,)), axis=-1).sum(axis=-1)  # off-board bits are 0
    valid = np.arange(64)[None, :] < np.asarray(rec["n_moves"]).astype(np.int64)[:, None]
    return valid & (board_size * board_size - discs <= empties)


def solve_record_winners(rec: dict, board_size: int, empties: int, rules: str = "reference", scoring: str = "reference",
                         device: int = 0) -> np.ndarray:
    """Per-position winner codes [G, 64] for training targets: every recorded position (before its move) with at most
    `empties` empty squares gets the winner under perfect play from there (engine.solve_endgame ->
    engine.perfect_play_winner); every other entry keeps its game's winner.  The record arrays are not changed."""
    n = board_size
    winners = np.repeat(np.asarray(rec["winner"]).astype(np.int32)[:, None], 64, axis=1)
    black, white = np.asarray(rec["black"], dtype=np.uint64), np.asarray(rec["white"], dtype=np.uint64)
    player = np.asarray(rec["player"]).astype(np.int64)
    sel = solvable_positions(rec, n, empties)
    if sel.any():
        own = np.where(player[sel] == 0, black[sel], white[sel])
        opp = np.where(player[sel] == 0, white[sel], black[sel])
        out = _e.solve_endgame(own, opp, board_size=n, max_empties=empties, device=device, rules=rules)
        winners[sel] = _e.perfect_play_winner(out["margin"], player[sel], scoring)
    return winners


# ---- RNG streams of episodes -------------------------------------------------------------------------------------
# The reference draws from CPython's process-global, time-seeded RNG, so no two episodes ever share randomness.  Here an
# episode's stream is keyed by (seed, game id) (include/oz_b200.h): by default the seed is drawn once per process from
# the OS and game ids come from a process-wide allocator, so consecutive calls, consecutive WorkerManager.run()s and
# different workers (one per GPU, INTEGRATION.md 1.1) never replay a stream.  Pass seed= / game_ids= for reproducible runs.
_PROCESS_SEED = int.from_bytes(os.urandom(8), "little")
_ids_lock = threading.Lock()
_next_game_id = 0


def allocate_game_ids(n: int) -> np.ndarray:
    """A block of n game ids never handed out before in this process."""
    global _next_game_id
    with _ids_lock:
        first = _next_game_id
        _next_game_id += int(n)
    return np.arange(first, first + int(n), dtype=np.uint64)


def execute_episodes(n_episodes, board_size, neural_network, degree_exploration, num_simulations, policy_temperature,
                     e_greedy, device: int = 0, seed: int | None = None, reference_aliasing: bool = False, game_ids=None,
                     max_concurrent: int = 4096, rules: str = "reference", scoring: str = "reference",
                     solve_empties: int = 0):
    """n_episodes x training.execute_episode as one GPU job; returns a list of example lists.  At most `max_concurrent`
    episodes are in flight (node pools are per slot); the others are queued on the device and start as slots free up.
    policy_temperature may be 0 (main.py:73-76 switches to it after `temperature_threshold` iterations).
    solve_empties > 0: the target z of every position with at most that many empties comes from the winner under perfect
    play (solve_record_winners), not from the game's outcome; not available with reference_aliasing."""
    if solve_empties and reference_aliasing:
        raise ValueError("solve_empties > 0 needs per-position targets, which reference_aliasing=True does not have")
    if seed is None:
        seed = _PROCESS_SEED
    if game_ids is None:
        game_ids = allocate_game_ids(n_episodes)
    sp = SelfPlay(board_size, neural_network, degree_exploration, max_games=min(n_episodes, max_concurrent),
                  num_simulations=num_simulations, device=device, seed=seed, rules=rules, scoring=scoring)
    try:
        rec = sp.play(n_episodes, policy_temperature, e_greedy, game_ids=game_ids)
    finally:
        sp.close()
    for g in range(n_episodes):
        logging.info(f'Episode finished: game {g}, winner channel {int(rec["winner"][g])}.')
    if reference_aliasing:
        return [records_to_examples(rec, g, board_size, True) for g in range(n_episodes)]
    winners = solve_record_winners(rec, board_size, solve_empties, rules, scoring, device) if solve_empties else None
    return records_to_examples_batch(rec, board_size, winners=winners)


def execute_episode(board_size, neural_network, degree_exploration, num_simulations, policy_temperature, e_greedy,
                    **kw):
    """Drop-in for training.execute_episode (training.py:26-27)."""
    return execute_episodes(1, board_size, neural_network, degree_exploration, num_simulations, policy_temperature,
                            e_greedy, **kw)[0]


# ---- workers.Worker plug-in (workers.py:18-79) --------------------------------------------------------------
class WorkType:
    EXECUTE_EPISODE = 'Execute Episode'
    DUEL_BETWEEN_NEURAL_NETWORKS = 'Duel between Neural Networks'
    EVALUATE_NEURAL_NETWORK = 'Evaluate Neural Network'


class Worker:
    """Mirror of workers.Worker's interface (workers.py:24-79) for use without the reference on sys.path."""

    def __init__(self):
        self._executor_thread = None
        self._results = None
        self._worker_manager = None

    def run(self, work_type, iterations, *args, **kwargs):
        self._results = []
        self._executor_thread = threading.Thread(name=self.get_executor_thread_name(), target=self._run,
                                                 args=(work_type, iterations, args, kwargs))
        self._executor_thread.start()

    def wait(self):
        return self._executor_thread.join() if self._executor_thread else None

    def get_results(self):
        return self._results

    def get_executor_thread_name(self):
        return f'{self.__class__.__name__}-{str(uuid.uuid4()).split("-", 1)[0]}'


def make_b200_worker(worker_base=Worker, device: int = 0, seed: int | None = None, rules: str = "reference",
                     scoring: str = "reference"):
    """Builds a ``B200Worker`` class deriving from ``worker_base`` — pass the reference's ``workers.Worker`` so that
    ``WorkerManager.add_worker``'s isinstance check (workers.py:186-190) accepts it.  seed=None (default): the
    process-wide OS-drawn seed; game ids always come from the process-wide allocator, so every run() of every worker
    plays episodes nobody has played before (see allocate_game_ids).  ``rules`` and ``scoring`` are the rule set and the
    scoring of every work type."""
    _e.board_arg(8, rules, scoring)  # unknown rule sets / scorings fail here, not in the worker thread

    class B200Worker(worker_base):
        def __init__(self):
            super().__init__()
            self.device = device
            self.seed = seed
            self.rules = rules
            self.scoring = scoring

        def _run(self, work_type, iterations, args, kwargs):
            # workers.py:57-65 runs the target once per iteration; here all iterations are one GPU batch and
            # _results still receives one entry per iteration (workers.py:54-55,180-184).
            # (the reference compares work types with `is`, workers.py:72-79; equal strings from another module's
            # WorkType class must match too, hence ==)
            if work_type == WorkType.EXECUTE_EPISODE:
                logging.info(f'Task {work_type}: {iterations} episodes as one GPU job on cuda:{self.device}')
                results = execute_episodes(iterations, *args, device=self.device, seed=self.seed, rules=self.rules,
                                           scoring=self.scoring, **kwargs)
            elif work_type == WorkType.DUEL_BETWEEN_NEURAL_NETWORKS:
                from . import arena
                logging.info(f'Task {work_type}: {iterations} duels as one GPU batch on cuda:{self.device}')
                results = arena.duels_between_neural_networks(iterations, *args, device=self.device, rules=self.rules,
                                                              scoring=self.scoring, **kwargs)
            elif work_type == WorkType.EVALUATE_NEURAL_NETWORK:
                from . import arena
                logging.info(f'Task {work_type}: {iterations} evaluations as one GPU batch on cuda:{self.device}')
                results = arena.evaluate_neural_network(*args, device=self.device, repeats=iterations,
                                                        rules=self.rules, scoring=self.scoring, **kwargs)
                results = results if isinstance(results, list) else [results]
            else:
                raise TypeError('expecting WorkType object')
            self._results.extend(results)

        def execute_episode(self, *args, **kwargs):
            return execute_episode(*args, device=self.device, seed=self.seed, rules=self.rules, scoring=self.scoring,
                                   **kwargs)

        def duel_between_neural_networks(self, *args, **kwargs):
            from . import arena
            return arena.duels_between_neural_networks(1, *args, device=self.device, rules=self.rules,
                                                       scoring=self.scoring, **kwargs)[0]

        def evaluate_neural_network(self, *args, **kwargs):
            from . import arena
            return arena.evaluate_neural_network(*args, device=self.device, rules=self.rules, scoring=self.scoring,
                                                 **kwargs)

    return B200Worker


B200Worker = make_b200_worker()
