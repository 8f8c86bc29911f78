"""Search side of the drop-in: ``OthelloMCTS`` (othelo_mcts.py:9-88 over MCTS/__init__.py:19-187) backed by
the CUDA tree kernel.  Same constructor and method names as the reference:

    mcts = OthelloMCTS(board_size, neural_network, degree_exploration)
    mcts.simulate(state, player)                         # othelo_mcts.py:22-26
    mcts.get_policy_action_probabilities(state, T)       # othelo_mcts.py:51-67
    mcts.get_state_actions(state)                        # othelo_mcts.py:40-41
    mcts.N(state, action=None)                           # MCTS/__init__.py:73-84

``neural_network`` may be
  * a ``B200NNet``            -> priors come from the on-device tcgen05 tower (OZ_PRIOR_NET);
  * a ``HashPriorNet``        -> closed-form priors evaluated inside the tree kernel (OZ_PRIOR_HASH);
  * anything with ``.predict`` (e.g. the reference's Keras NNetWrapper) -> leaves are handed to the host and
    ``predict`` is called once per expanded node, exactly as the reference does (OZ_PRIOR_HOST).
Aliases ``search`` / ``getActionProb`` are the alpha-zero-general names used in BASELINE.json.
``rules="standard"`` searches under standard Othello flipping instead of the reference's flip rule, and
``scoring="standard"`` values a drawn terminal as 0 instead of as a BLACK win.  ``values="standard"`` negates a child's
value only when the move swapped the side to move, and ``solve_leaves=K`` (with standard values and scoring) solves new
leaves with at most K empties exactly (``engine.Engine``).  ``dirichlet_alpha`` > 0 mixes Dirichlet noise into each
root's priors once, with weight ``dirichlet_fraction`` (the root exploration of ``engine.Engine``).  The noise stream is
keyed by (seed, game id, root position); by default every instance takes the process-wide OS-drawn seed and a game id
nobody has used before (``selfplay.allocate_game_ids``), so a new instance per episode, as the reference's training loop
builds them, explores differently every time.  Pass ``seed=`` and ``game_id=`` for a reproducible search.
"""
from __future__ import annotations

import random

import numpy as np

from . import engine as _e
from .net import B200NNet, NeuralNets, bits_to_board
from .othello import OthelloGame, OthelloPlayer, _bits, game_class


class HashPriorNet:
    """Deterministic stand-in network (SURVEY Appendix B.3); evaluated on the device by the tree kernel."""
    network_type = NeuralNets.ONN

    def predict(self, board):  # pragma: no cover - the device evaluates it; kept for interface completeness
        raise NotImplementedError("HashPriorNet is evaluated inside the CUDA tree kernel")


class OthelloMCTS:
    def __init__(self, board_size, neural_network, degree_exploration, nodes: int = 65536, device: int = 0,
                 rules: str = "reference", scoring: str = "reference", values: str = "reference",
                 solve_leaves: int = 0, dirichlet_alpha: float = 0.0, dirichlet_fraction: float = 0.25,
                 seed: int | None = None, game_id: int | None = None):
        self._board_size = board_size
        self._neural_network = neural_network
        self.degree_explorarion = degree_exploration  # (sic) MCTS/__init__.py:27
        if getattr(neural_network, "network_type", NeuralNets.ONN) not in (NeuralNets.ONN, "ONN") and \
                getattr(getattr(neural_network, "network_type", None), "name", "ONN") != "ONN":
            raise TypeError("only the two-channel ONN board view is implemented on the B200 path")
        if isinstance(neural_network, HashPriorNet):
            mode = _e.PRIOR_HASH
        elif isinstance(neural_network, B200NNet):
            mode = _e.PRIOR_NET
        else:
            mode = _e.PRIOR_HOST
        self._mode = mode
        from . import selfplay  # the process-wide seed and game-id allocator (selfplay imports this module)
        self.seed = selfplay._PROCESS_SEED if seed is None else int(seed)
        self.game_id = int(selfplay.allocate_game_ids(1)[0]) if game_id is None else int(game_id)
        self._eng = _e.Engine(board_size, max_games=1, nodes_per_game=nodes, prior_mode=mode,
                              c_puct=float(degree_exploration), seed=self.seed, device=device, rules=rules,
                              scoring=scoring, values=values, solve_leaves=solve_leaves,
                              dirichlet_alpha=dirichlet_alpha, dirichlet_fraction=dirichlet_fraction)
        self._game = game_class(rules, scoring)
        if mode == _e.PRIOR_NET:
            self._eng.load_weights(neural_network.blob, neural_network.channels, neural_network.precision)
        self._eng.reset(1, game_ids=[self.game_id])
        self._root = None

    # -- helpers ------------------------------------------------------------------------------------
    def _set_root(self, black, white, player):
        key = (black, white, player)
        if key != self._root:
            self._eng.set_roots([black], [white], [player])
            self._root = key

    def _predict_batch(self, own, opp):
        n = self._board_size
        pis, vs = [], []
        for o, p in zip(own, opp):
            pi, v = self._neural_network.predict(bits_to_board(o, p, n))
            pis.append(np.asarray(pi, dtype=np.float32).reshape(-1))
            vs.append(np.float32(v))
        return np.stack(pis), np.array(vs, dtype=np.float32)

    def _canonical_root(self, state):
        ch0, ch1 = _bits(state)
        self._set_root(ch0, ch1, 0)

    # -- reference API --------------------------------------------------------------------------------
    def simulate(self, state, player, num_simulations: int = 1):
        """One simulation from ``state`` with ``player`` to move (othelo_mcts.py:22-26). ``num_simulations`` > 1
        runs that many sequential simulations in one launch (same result as calling it repeatedly)."""
        black, white = _bits(state)
        self._set_root(black, white, 0 if player is OthelloPlayer.BLACK or player == 0 else 1)
        self._eng.search(num_simulations, self._predict_batch if self._mode == _e.PRIOR_HOST else None)

    def N(self, state, action=None):
        self._canonical_root(state)
        v, ns = self._eng.visits()
        if action is None:
            return int(ns[0])
        return int(v[0][int(action[0]) * 8 + int(action[1])])

    def get_state_actions(self, state):
        return [tuple(int(x) for x in a) for a in OthelloGame.get_player_valid_actions(state, OthelloPlayer.BLACK)]

    def is_terminal_state(self, state):
        return OthelloGame.has_board_finished(state)

    def get_state_reward(self, state):
        winner = self._game.get_board_winning_player(state)[0]
        return 0 if winner is None else winner.value  # None: a draw under standard scoring

    def get_next_state(self, state, action):
        board = np.copy(state)
        self._game.flip_board_squares(board, OthelloPlayer.BLACK, *action)
        if OthelloGame.has_player_actions_on_board(board, OthelloPlayer.WHITE):
            board = OthelloGame.invert_board(board)
        return board

    def get_policy_action_probabilities(self, state, temperature):
        n = self._board_size
        self._canonical_root(state)
        v, _ = self._eng.visits()
        counts = np.zeros((n, n))
        for r in range(n):
            for c in range(n):
                counts[r, c] = v[0][r * 8 + c]
        if temperature == 0:
            bests = np.argwhere(counts == counts.max())
            row, col = random.choice(bests)
            probabilities = np.zeros((n, n))
            probabilities[row, col] = 1
            return probabilities
        probabilities = np.zeros((n, n))
        legal = self.get_state_actions(state)
        for (r, c) in legal:
            probabilities[r, c] = int(counts[r, c]) ** (1 / temperature)
        return probabilities / (np.sum(probabilities) or 1)

    # alpha-zero-general names (SURVEY Appendix D)
    search = simulate
    getActionProb = get_policy_action_probabilities

    def close(self):
        self._eng.close()
