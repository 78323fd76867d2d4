"""Single-game interactive API in the shape of the reference's play.py PlayTensor (:11-91), the backend of its Streamlit GUI
(SURVEY.md 8f rank 4; a "next" row): one game, the network picks the arg-max move of a `num_searches`-simulation search.
Thin host-side wrapper over the same drop-in classes (ChessTensor / MCTS0 / policyNN -> libszb200)."""
import torch

from . import chess_compat as chess
from .chess_tensor import ChessTensor
from .mcts import MCTS0
from .network import policyNN


class PlayTensor:
    def __init__(self, model_path=None, num_searches=200, C=2, chess960=False, precision="bf16", leaves_per_tree=1, eval_cache_slots=0):
        """leaves_per_tree > 1: the opt-in multi-leaf search (virtual loss; ~7x faster move decisions for a single game at 8, but
        not the reference's visit counts).  eval_cache_slots > 0 (a power of two in [64, 65536]): the exact evaluation cache, so
        positions the previous move's search evaluated skip the network (the same moves)."""
        self.args = {"C": C, "num_searches": num_searches, "leaves_per_tree": leaves_per_tree, "eval_cache_slots": eval_cache_slots}
        self.chess960 = chess960
        self.network = policyNN({"precision": precision})
        if model_path:                                    # play.py:25-28: torch.load(..., map_location) -> load_state_dict
            self.network.load_state_dict(torch.load(model_path, map_location="cpu"))
        self.network.eval()
        self.start_new_game()

    def start_new_game(self):
        self.game = ChessTensor(chess960=self.chess960)
        self.board = self.game.board
        self.mcts = MCTS0(game=self.game, model=self.network, args=self.args)

    def get_best_move(self):
        """play.py:40-43: arg-max of the visit fractions (first maximum = lowest move index on ties)"""
        probs = self.mcts.search(self.board, verbose=False)
        return max(probs, key=probs.get)

    def move(self, move):
        if isinstance(move, str):
            move = chess.Move.from_uci(move)
        self.game.move_piece(move)                        # raises ValueError("Invalid move") like the reference

    def model_move(self):
        m = self.get_best_move()
        self.game.move_piece(m)
        return m

    def check_if_end(self):
        value, terminated = self.game.get_value_and_terminated()
        if not terminated:
            return None
        return "draw" if value == 0 else ("black" if self.board.turn else "white")
