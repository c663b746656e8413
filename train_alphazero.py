#!/usr/bin/env python
"""CLI with the reference's flags (train_alphazero.py:30-61) for all three modes:

    python train_alphazero.py --mode self-play --rows 8 --cols 8 --simulations 800 --episodes 4096
    python train_alphazero.py --mode evaluate  --simulations 100

``--mode self-play`` -> generate_self_play_data (train_alphazero.py:103-122); ``--mode evaluate`` -> 10 games
AlphaZeroPlayer vs RandomPlayer with alternating colours (:124-243); ``--mode train`` -> AlphaZero.run (:86-101): per
iteration self-play with the best model, the CUDA learner on the data directory, current-vs-best arena, promotion at a
win ratio >= 0.6 -- every stage on the GPU.  Extra flags: ``--rules-rowcol`` (browser-game row/column rule),
``--init-model`` (write a randomly initialised checkpoint if none exists), ``--arena-games`` (default 40).
"""
import argparse
import logging
import os
import sys

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
logging.basicConfig(level=logging.INFO, format="%(asctime)s - %(name)s - %(levelname)s - %(message)s")
logger = logging.getLogger("AlphaZeroTraining")


def parse_args(argv=None):
    p = argparse.ArgumentParser(description="Yin-Yang AlphaZero (B200 self-play engine)")
    p.add_argument("--rows", type=int, default=8)
    p.add_argument("--cols", type=int, default=8)
    p.add_argument("--iterations", type=int, default=100)
    p.add_argument("--episodes", type=int, default=100)
    p.add_argument("--simulations", type=int, default=800)
    p.add_argument("--epochs", type=int, default=10)
    p.add_argument("--batch-size", type=int, default=64)
    p.add_argument("--lr", type=float, default=0.001)
    p.add_argument("--workers", type=int, default=1)
    p.add_argument("--mcts-threads", type=int, default=1)
    p.add_argument("--model-dir", type=str, default="models")
    p.add_argument("--data-dir", type=str, default="data")
    p.add_argument("--resume", action="store_true")
    p.add_argument("--mode", choices=["train", "self-play", "evaluate"], default="train")
    p.add_argument("--output-model", type=str, default="best_model.pth.tar")
    p.add_argument("--rules-rowcol", action="store_true", help="also apply the browser game's row/column rule")
    p.add_argument("--init-model", action="store_true", help="create a randomly initialised model file if missing")
    p.add_argument("--eval-games", type=int, default=10)
    p.add_argument("--arena-games", type=int, default=40, help="--mode train: games of current vs best per iteration (alphazero.py:136)")
    p.add_argument("--file-loop", action="store_true",
                   help="--mode train: exchange self-play data and weights between the stages through files in --data-dir / "
                        "--model-dir like the reference, instead of keeping the examples on the GPU(s)")
    p.add_argument("--replay-wire", choices=["arrays", "native", "reference"], default="arrays",
                   help="'arrays' (default): boards as one int8[N,n,m] array under the reference's npz keys; 'native': an object "
                        "array of this package's YinYangLogic; 'reference': boards pickled as "
                        "src.yin_yang.yin_yang_logic.YinYangLogic so that the reference's own trainer loads the .npz "
                        "without this package")
    p.add_argument("--eval-symmetry", choices=["none", "random", "average"], default="none",
                   help="network evaluation of the search leaves in every mode: as they are (default), in one dihedral form "
                        "of the board hashed from the position and the seed, or averaged over all forms (8x the network FLOPs)")
    p.add_argument("--full-search-prob", type=float, default=1.0,
                   help="self-play playout cap randomisation (--mode self-play / train): the share of moves that get the full "
                        "--simulations search and become training examples; the others get a fast search that only advances "
                        "the game (default 1: every move)")
    p.add_argument("--fast-simulations", type=int, default=None,
                   help="simulations of a fast self-play search when --full-search-prob < 1 (default: --simulations)")
    return p.parse_args(argv)


def main(argv=None):
    args = parse_args(argv)
    import yy_b200  # noqa: F401
    from yinyang_game_alphazero_b200.game import YinYangGame, RULE_ROWCOL
    from yinyang_game_alphazero_b200.network import YinYangNeuralNetwork
    from yinyang_game_alphazero_b200.players import AlphaZeroPlayer, RandomPlayer
    from yinyang_game_alphazero_b200.self_play import generate_self_play_data

    game = YinYangGame(n=args.rows, m=args.cols, rule_flags=RULE_ROWCOL if args.rules_rowcol else 0)
    for d in (args.model_dir, args.data_dir):
        os.makedirs(d, exist_ok=True)
    model_path = os.path.join(args.model_dir, args.output_model)
    if args.mode == "train":                                             # train_alphazero.py:86-101
        from yinyang_game_alphazero_b200.alphazero import AlphaZero
        world = int(os.environ.get("WORLD_SIZE", "1"))
        if world > 1:                                                    # torchrun: one process per GPU
            import torch
            import torch.distributed as dist
            local = int(os.environ.get("LOCAL_RANK", "0"))
            torch.cuda.set_device(local)
            dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        az = AlphaZero(game=game, model_dir=args.model_dir, data_dir=args.data_dir, num_iterations=args.iterations,
                       num_episodes=args.episodes, num_simulations=args.simulations, num_epochs=args.epochs,
                       num_workers=args.workers, mcts_threads=args.mcts_threads, eval_games=args.arena_games,
                       batch_size=args.batch_size, lr=args.lr, eval_symmetry=args.eval_symmetry,
                       full_search_prob=args.full_search_prob, fast_simulations=args.fast_simulations)
        if args.file_loop:
            az.run()                                                     # the reference's loop: data files between the stages
        else:
            az.run_device_resident()                                     # examples stay on the GPU(s); NCCL gather / broadcast
        if world > 1:
            dist.destroy_process_group()
        logger.info("Training completed!")
        return 0
    if not os.path.exists(model_path):
        if args.init_model:
            YinYangNeuralNetwork(game).save_model(model_path)
            logger.info(f"Wrote randomly initialised model to {model_path}")
        else:
            logger.error(f"Model file not found: {model_path}")          # train_alphazero.py:107-109
            return 1
    if args.mode == "self-play":
        logger.info(f"Generating self-play data using model: {model_path}")
        world = int(os.environ.get("WORLD_SIZE", "1"))
        if world > 1:
            # torchrun, one process per GPU (the counterpart of the reference's --workers processes, self_play.py:288-335):
            # the episodes are sharded over the ranks, the examples gathered to rank 0 over NCCL, ONE file is written
            from yinyang_game_alphazero_b200.self_play import generate_self_play_data_distributed
            data_file = generate_self_play_data_distributed(game=game, model_path=model_path, output_dir=args.data_dir,
                                                            num_games=args.episodes, num_simulations=args.simulations,
                                                            wire=args.replay_wire, eval_symmetry=args.eval_symmetry,
                                                            full_search_prob=args.full_search_prob,
                                                            fast_simulations=args.fast_simulations)
        else:
            data_file = generate_self_play_data(game=game, model_path=model_path, output_dir=args.data_dir,
                                                num_games=args.episodes, num_workers=args.workers,
                                                num_simulations=args.simulations, wire=args.replay_wire,
                                                eval_symmetry=args.eval_symmetry, full_search_prob=args.full_search_prob,
                                                fast_simulations=args.fast_simulations)
        if data_file:
            logger.info(f"Self-play data generation completed. Data saved to {data_file}")
        return 0
    # evaluate: AlphaZero vs random, colours alternate (train_alphazero.py:165-243)
    az = AlphaZeroPlayer(game=game, model_path=model_path, num_simulations=args.simulations, num_threads=args.mcts_threads,
                         eval_symmetry=args.eval_symmetry)
    rnd = RandomPlayer(game, verbose=False)
    az_wins = rnd_wins = draws = 0
    for i in range(args.eval_games):
        az.reset()
        board, player = game.getInitBoard(), 1
        first_is_az = (i % 2 == 0)
        first, second = (az, rnd) if first_is_az else (rnd, az)
        while True:
            action = (first if player == 1 else second).play(board, player)
            if action == -1:
                break                                                     # no result recorded, like the reference (:198-200)
            board, player = game.getNextState(board, player, action)
            result = game.getGameEnded(board, player)
            if result != 0:
                if result == 1:
                    az_wins, rnd_wins = (az_wins + 1, rnd_wins) if first_is_az else (az_wins, rnd_wins + 1)
                elif result == -1:
                    az_wins, rnd_wins = (az_wins, rnd_wins + 1) if first_is_az else (az_wins + 1, rnd_wins)
                else:
                    draws += 1
                break
        black, white = board.count_pieces()
        logger.info(f"Game {i + 1} finished. Score: Black={black}, White={white}")
    logger.info(f"Evaluation completed. AlphaZero wins: {az_wins}, Random wins: {rnd_wins}, Draws: {draws}")
    logger.info(f"AlphaZero win rate: {az_wins / max(1, args.eval_games):.2f}")
    return 0


if __name__ == "__main__":
    sys.exit(main())
