"""Drop-in for the reference's mcts.py: MCTS0.search returns {move: visit fraction} over all root children in
ascending policy-index order (mcts.py:113-122).  The whole search -- PUCT descent, move generation, plane
encoding, network, masking/normalisation/noise, expansion, backup -- runs in libszb200 (szb_search)."""
import numpy as np
import torch

from . import chess_compat as chess
from . import runtime
from .chess_tensor import ChessTensor, index_move
from .mctsnode import tree_view


class MCTS0:
    def __init__(self, game=None, args=None, model=None):
        self.game = game
        self.args = args
        self.model = model
        self.root = None

    @torch.no_grad()
    def search(self, state, verbose=True, learning=False):
        args = self.args
        n = int(args['num_searches'])
        eng = runtime.get_engine(min_games=1, min_searches=n, leaves_per_tree=runtime.leaves_of(args))
        runtime.sync_weights(eng, self.model)
        explore = runtime.exploration_of(args)
        cache_slots = runtime.eval_cache_of(args)
        eng = self.game._engine()                    # replays the game into slot 0 if another game was there
        eng.set_exploration(seed=int(args.get('seed', 0)), **explore)
        eng.set_eval_cache(cache_slots)
        white = bool(state.turn)
        eng.search(n, float(args['C']), bool(learning), runtime.evaluator_of(self.model),
                   want_visits=False, want_children=False)
        idx, vis, cnt = eng.root_children()
        k = int(cnt[0])
        self._engine = eng
        self._white = white
        counts = vis[0, :k].astype(np.int64)
        total = int(counts.sum())
        legal = {m.uci(): m for m in self.game.board.legal_moves}
        action_probs = {}
        for i, c in zip(idx[0, :k], counts):
            m = index_move(int(i), white)
            m = legal.get(m.uci() + "q", legal.get(m.uci(), m))       # queen promotions carry their piece
            action_probs[m] = int(c) / total                        # ZeroDivisionError when num_searches == 1, as in the reference
        return action_probs

    def tree(self):
        """mctsnode.Node view of the last search's tree (root first)."""
        export = self._engine.tree_export(0)
        return tree_view(export, self.args, self._white, lambda i, color: index_move(i, color))
