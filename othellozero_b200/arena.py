"""Arena ("next" row, SURVEY §8f rank 2): agents and duels of agents.py:11-84 on top of the CUDA engine.

* ``OthelloAgent`` / ``RandomOthelloAgent`` / ``NeuralNetworkOthelloAgent`` / ``duel_between_agents`` mirror the
  reference game by game (same names, same semantics: the network agent always plays at temperature 0 with
  ``random.choice`` over the arg-max set, agents.py:44-68, othelo_mcts.py:54-62).
* ``pit`` plays many games at once, network vs network or network vs the random agent: one engine per network side
  (each agent keeps its own tree for the whole game, agents.py:49), one search launch per move for all games whose
  turn it is.
* ``duels_between_neural_networks`` / ``evaluate_neural_network`` are the batched forms of the worker work types
  (workers.py:18-21); ``selfplay.B200Worker`` dispatches all three work types.

The reference's own drivers ``training.duel_between_neural_networks`` / ``evaluate_neural_network`` are broken
(SURVEY §0.8); ``pit`` follows the working semantics of main.py:165-197 (who won, counted per game).
``rules="standard"`` plays every game of a batched driver under standard Othello flipping; the per-game agents take the
rule set from their game (``othello.StandardOthelloGame``).  ``scoring="standard"`` scores a game with equal disc counts
as a draw (winner code 2, no win for either side) in the search and in the result; the per-game agents take it from
their game too (``othello.game_class``).
"""
from __future__ import annotations

import random

import numpy as np

from . import engine as _e
from ._lib import WINNER_DRAW
from .mcts import HashPriorNet, OthelloMCTS
from .net import B200NNet
from .othello import BoardView, OthelloGame, OthelloPlayer


class OthelloAgent:
    def __init__(self, game):
        self.game = game

    def play(self):
        raise NotImplementedError


class RandomOthelloAgent(OthelloAgent):
    """agents.py:20-24."""

    def play(self):
        possible_moves = tuple(self.game.get_valid_actions())
        move = random.choice(possible_moves)
        self.game.play(*move)


class NeuralNetworkOthelloAgent(OthelloAgent):
    """agents.py:44-68 (temperature is forced to 0 there, :46)."""

    def __init__(self, game, neural_network, num_simulations, degree_exploration, temperature=0):
        self.temperature = 0
        self.neural_network = neural_network
        self.num_simulations = num_simulations
        self.mcts = OthelloMCTS(game.board_size, neural_network, degree_exploration, rules=game.rules,
                                scoring=game.scoring)
        super().__init__(game)

    def play(self):
        state = self.game.board(BoardView.TWO_CHANNELS)
        self.mcts.simulate(state, self.game.current_player, num_simulations=self.num_simulations)
        if self.game.current_player == OthelloPlayer.WHITE:
            state = OthelloGame.invert_board(state)
        action_probabilities = self.mcts.get_policy_action_probabilities(state, self.temperature)
        valid_actions = self.game.get_valid_actions()
        best_action = max(valid_actions, key=lambda position: action_probabilities[tuple(position)])
        self.game.play(*best_action)


def duel_between_agents(game, agent_1, agent_2):
    """agents.py:71-84: agent_1 is BLACK, agent_2 WHITE; returns (winning agent, points), the agent None for a draw
    under standard scoring."""
    players_agents = {OthelloPlayer.BLACK: agent_1, OthelloPlayer.WHITE: agent_2}
    while not game.has_finished():
        players_agents[game.current_player].play()
    winner, points = game.get_winning_player()
    return players_agents.get(winner), points


RANDOM_AGENT = "random"   # a side of pit() that plays RandomOthelloAgent's policy (agents.py:20-24)


def _mode_for(net):
    if isinstance(net, HashPriorNet):
        return _e.PRIOR_HASH
    if isinstance(net, B200NNet):
        return _e.PRIOR_NET
    raise TypeError("pit() needs B200NNet / HashPriorNet agents (or RANDOM_AGENT)")


def _popcount(x: np.ndarray) -> np.ndarray:
    return np.unpackbits(np.ascontiguousarray(x, dtype="<u8").view(np.uint8).reshape(-1, 8), axis=1).sum(axis=1).astype(np.int64)


def _kth_set_bits(masks: np.ndarray, k: np.ndarray) -> np.ndarray:
    """Square (bit index) of the k[i]-th set bit of masks[i], ascending = row-major; all games at once."""
    bits = np.unpackbits(np.ascontiguousarray(masks, dtype="<u8").view(np.uint8).reshape(-1, 8), axis=1,
                         bitorder="little").astype(bool)                       # [G, 64], column = square bit
    rank = np.cumsum(bits, axis=1) - 1
    return np.argmax(bits & (rank == np.asarray(k, dtype=np.int64)[:, None]), axis=1).astype(np.int32)


def _draw_indices(rng, counts: np.ndarray) -> np.ndarray:
    """One uniform index in [0, counts[i]) per game.  A numpy Generator draws them all at once; any other rng (Python's
    ``random`` by default, as in the reference: agents.py:22-23, othelo_mcts.py:58-59) is asked once per game that
    really has a choice, with the reference's call form ``rng.choice(sequence)``."""
    counts = np.asarray(counts, dtype=np.int64)
    if hasattr(rng, "integers"):
        return rng.integers(0, counts)
    out = np.zeros(counts.shape[0], dtype=np.int64)
    for i in np.nonzero(counts > 1)[0]:
        out[i] = rng.choice(range(int(counts[i])))
    return out


def pit(board_size, net_black, net_white, num_simulations, degree_exploration=1, n_games=64, device=0, rng=None,
        start_black=None, start_white=None, start_player=None, rules="reference", scoring="reference"):
    """n_games simultaneous duels, net_black playing BLACK.  Returns dict(winner [n_games] 0/1, black, white, plies,
    points, draws [n_games] bool: equal final counts).  Under reference scoring a draw is a BLACK win (winner 0); under
    ``scoring="standard"`` its winner is 2, and both searches value drawn terminals as 0.
    Every step is one kernel chain over all games whose turn it is: one search launch per network side
    (NeuralNetworkOthelloAgent.play, agents.py:52-68, always temperature 0), one move-generator launch for a
    ``RANDOM_AGENT`` side (RandomOthelloAgent.play, agents.py:20-24; main.py:165-197 evaluates the network against it),
    one rules launch to apply the moves.  Ties in the visit counts and the random agent's moves are drawn from ``rng``
    (Python's ``random`` like the reference, or a numpy Generator for fully vectorised draws) over the candidates in
    row-major order.  Both sides search, and every move is applied, under ``rules``."""
    _e.board_arg(board_size, rules, scoring)
    rng = rng or random
    n = board_size
    nodes = num_simulations * (n * n) + 64
    engines = []
    for net in (net_black, net_white):
        if isinstance(net, str) and net == RANDOM_AGENT:
            engines.append(None)
            continue
        mode = _mode_for(net)
        e = _e.Engine(n, max_games=n_games, nodes_per_game=nodes, prior_mode=mode, c_puct=float(degree_exploration),
                      device=device, rules=rules, scoring=scoring)
        if mode == _e.PRIOR_NET:
            e.load_weights(net.blob, net.channels, net.precision)
        engines.append(e)
    if start_black is None:
        from .othello import _bits
        bb, ww = _bits(OthelloGame.initial_board(n))
        black = np.full(n_games, bb, dtype=np.uint64)
        white = np.full(n_games, ww, dtype=np.uint64)
        player = np.zeros(n_games, dtype=np.int32)
    else:
        black = np.array(start_black, dtype=np.uint64)
        white = np.array(start_white, dtype=np.uint64)
        player = np.array(start_player, dtype=np.int32)
    for e in engines:
        if e is not None:
            e.reset(n_games, black, white, player)
    finished = np.zeros(n_games, dtype=bool)
    plies = np.zeros(n_games, dtype=np.int32)
    try:
        while not finished.all():
            for side, e in enumerate(engines):
                turn = (~finished) & (player == side)
                if not turn.any():
                    continue
                idx = np.nonzero(turn)[0]
                own = np.where(player[idx] == 0, black[idx], white[idx])
                opp = np.where(player[idx] == 0, white[idx], black[idx])
                if e is None:  # the random agent: uniform over the legal moves (GPU move generator, host RNG)
                    legal = _e.legal_moves(own, opp, n, device)
                    sq = _kth_set_bits(legal, _draw_indices(rng, _popcount(legal)))
                else:
                    # games where it is not this agent's turn get a root with no legal move for the mover: the
                    # kernel skips them (0 simulations), exactly like an agent that is not asked to play
                    e.set_roots(np.where(turn, black, 0).astype(np.uint64), np.where(turn, white, 0).astype(np.uint64), player)
                    e.search(num_simulations)
                    visits = e.visits()[0][idx]                                    # [games to move, 64] by square bit
                    tied = visits == visits.max(axis=1, keepdims=True)             # othelo_mcts.py:58: the arg-max set
                    pick = _draw_indices(rng, tied.sum(axis=1))                    # a unique maximum needs no draw
                    sq = np.argmax(tied & ((np.cumsum(tied, axis=1) - 1) == pick[:, None]), axis=1).astype(np.int32)
                o2, p2, fl, _ = _e.apply_moves(own, opp, sq, n, device, rules=rules)
                assert not (fl & 0x80000000).any()
                swapped = (fl & 1).astype(bool)
                npl = np.where(swapped, 1 - player[idx], player[idx]).astype(np.int32)
                black[idx] = np.where(npl == 0, o2, p2)
                white[idx] = np.where(npl == 0, p2, o2)
                player[idx] = npl
                plies[idx] += 1
                finished[idx] = (fl & 4) != 0
    finally:
        for e in engines:
            if e is not None:
                e.close()
    cb, cw = _e.score(black, white, device)
    draws = cb == cw
    winner = np.where(cb >= cw, 0, 1)
    if scoring == "standard":
        winner = np.where(draws, WINNER_DRAW, winner)
    return dict(winner=winner, black=black, white=white, plies=plies, points=np.maximum(cb, cw), draws=draws)


# ---- batched arena drivers (the worker work types of workers.py:18-21,72-79) -----------------------------------------
def duels_between_neural_networks(n_duels, board_size, neural_network_1, neural_network_2, degree_exploration,
                                  num_simulations, device=0, rng=None, rules="reference", scoring="reference"):
    """``n_duels`` x training.duel_between_neural_networks (training.py:75-89) as one batch: network 1 plays BLACK
    (agent_1 of duel_between_agents, agents.py:71-74); each entry is 0 if network 1 won, 1 if network 2 won, and 2 for a
    draw under standard scoring."""
    out = pit(board_size, neural_network_1, neural_network_2, num_simulations, degree_exploration, n_games=n_duels,
              device=device, rng=rng, rules=rules, scoring=scoring)
    return [int(w) for w in out["winner"]]


def evaluate_neural_network(board_size, total_iterations, neural_network, num_simulations, degree_exploration,
                            agent_class=RandomOthelloAgent, agent_arguments=(), device=0, rng=None, repeats=1,
                            rules="reference", scoring="reference"):
    """training.evaluate_neural_network (training.py:92-115) with the working semantics of main.py:165-197: the network
    meets ``agent_class`` (RandomOthelloAgent) in ``total_iterations`` games, colours shuffled per game; returns the
    network's wins (a draw under standard scoring is not a win).  ``repeats`` > 1 plays that many evaluations in the
    same batch and returns a list of win counts."""
    if agent_class is not RandomOthelloAgent:
        raise TypeError("the batched evaluation plays against RandomOthelloAgent (main.py:165-197)")
    _e.board_arg(board_size, rules, scoring)
    rng = rng or random
    games = total_iterations * repeats
    net_is_black = np.array([rng.random() < 0.5 for _ in range(games)], dtype=bool)   # random.shuffle of two agents
    net_won = np.zeros(games, dtype=bool)
    for black_side in (True, False):
        sel = np.nonzero(net_is_black == black_side)[0]
        if sel.size == 0:
            continue
        a, b = (neural_network, RANDOM_AGENT) if black_side else (RANDOM_AGENT, neural_network)
        out = pit(board_size, a, b, num_simulations, degree_exploration, n_games=int(sel.size), device=device, rng=rng,
                  rules=rules, scoring=scoring)
        net_won[sel] = out["winner"] == (0 if black_side else 1)
    wins = net_won.reshape(repeats, total_iterations).sum(axis=1)
    return int(wins[0]) if repeats == 1 else [int(w) for w in wins]
