"""The GUI's AI-move endpoint without the web server (SURVEY 8f-4): the body of ``POST /api/ai_move``
(src/gui/server.py:30-129) as a function -- same request fields (``board``, ``currentPlayer``, ``rows``, ``cols``,
``modelPath``) and the same response dictionaries (``{'validMove': True, 'row', 'col'}``, ``{'validMove': False,
'message'}``, ``{'error'}``) -- on the batch-1 latency path of the engine (one game, 100 simulations, one persistent
kernel launch per move).  A Flask route is a one-liner on top: ``return jsonify(get_ai_move(request.json))``.
"""
from __future__ import annotations

import logging

import numpy as np

from .game import YinYangGame
from .players import AlphaZeroPlayer

logger = logging.getLogger("YinYangGUI")

_state = {"game": None, "player": None, "model_path": None}      # server.py:17-19 module globals


def get_ai_move(data, num_simulations=100, num_threads=1, eval_symmetry="none"):
    try:
        board_state, player = data.get("board"), data.get("currentPlayer")
        rows, cols = data.get("rows"), data.get("cols")
        model_path = data.get("modelPath", "models/best_model.pth.tar")
        game = _state["game"]
        if game is None or game.getBoardSize() != (rows, cols):
            game = _state["game"] = YinYangGame(rows, cols)
        az = _state["player"]
        if az is None or az.game.getBoardSize() != (rows, cols) or _state["model_path"] != model_path or az.mcts.num_threads != max(1, num_threads) \
                or az.mcts.eval_symmetry != eval_symmetry:
            try:
                az = _state["player"] = AlphaZeroPlayer(game=game, model_path=model_path, num_simulations=num_simulations, num_threads=num_threads,
                                                      eval_symmetry=eval_symmetry)
                _state["model_path"] = model_path
            except Exception as e:  # server.py:58-60
                logger.error(f"Error initializing AlphaZero player: {e}", exc_info=True)
                return {"error": f"Failed to initialize AlphaZero: {e}"}
        board = game.getInitBoard()
        board.board[:, :] = np.asarray(board_state, dtype=np.int8).reshape(rows, cols)
        valid_moves = game.getValidMoves(board, player)
        if np.sum(valid_moves) == 0:
            return {"validMove": False, "message": "No valid moves available"}
        try:
            az.reset()
            action = az.play(board, player)
            if action == -1:
                return {"validMove": False, "message": "No valid moves available"}
            if valid_moves[action] != 1:                          # server.py:100-113: random legal fallback
                idx = np.where(valid_moves == 1)[0]
                if len(idx) == 0:
                    return {"validMove": False, "message": "No valid moves available"}
                action = int(np.random.choice(idx))
            row, col = game._action_to_coords(action)
            return {"validMove": True, "row": int(row), "col": int(col)}
        except Exception as e:
            logger.error(f"Error getting AI move: {e}", exc_info=True)
            return {"error": f"Failed to get AI move: {e}"}
    except Exception as e:
        logger.error(f"Error processing AI move request: {e}", exc_info=True)
        return {"error": str(e)}
