"""Throughput of evaluation games on the device (SelfPlay.play_test_games against the expert), one JSON line per workload.

    python scripts/eval_throughput.py [--seconds 1.0] [--workloads tictactoe,connect4]

Workloads: TicTacToe, 8192 games per call, N = 25 (the config's value); Connect4, 1024 games per call, N = 200, the
default tensor-core towers (x3); both with muzero_player 0 and 1, on seeded synthetic weights.  One warm-up call, then
timed calls until at least --seconds have passed (a host clock around calls that end in a device synchronisation).
Reported: evaluation games/s, moves/s of both sides, positions searched/s (every slot searches at every batched move,
games played past the requested ids included), W/D/L of the timed calls, and the GPU's name and power limit read in
the same run.
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

WORKLOADS = {"tictactoe": (8192, 25), "connect4": (1024, 200)}


def gpu_info():
    out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True, check=True).stdout.strip()
    name, power = (x.strip() for x in out.split(",", 1))
    return name, power


def run(game, games, N, muzero_player, seconds):
    from muzero_general_b200 import self_play as sp
    from muzero_general_b200.games import load_game_module
    from muzero_general_b200.netspec import netspec_from_config, synthetic_weights
    mod = load_game_module(game)
    cfg = mod.MuZeroConfig()
    cfg.rng_mode, cfg.num_simulations, cfg.test_parallel_games = "philox", N, games
    worker = sp.SelfPlay({"weights": synthetic_weights(netspec_from_config(cfg), 0)}, mod.Game, cfg, seed=0)
    assert worker.loop_path == "device"
    worker.play_test_games(games, "expert", muzero_player)                    # warm-up: engine, graphs, loop
    calls = n_games = moves = searches = 0
    wins = draws = losses = 0
    t0 = time.perf_counter()
    while True:
        played, summary = worker.play_test_games(games, "expert", muzero_player)
        calls += 1
        n_games += len(played)
        moves += played.total_moves
        searches += worker.last_test_searches
        wins, draws, losses = wins + summary["wins"], draws + summary["draws"], losses + summary["losses"]
        elapsed = time.perf_counter() - t0
        if elapsed >= seconds:
            break
    worker.close()
    worker._test_model.engine.close()
    return dict(game=game, games_per_call=games, num_simulations=N, opponent="expert", muzero_player=muzero_player,
                calls=calls, seconds=round(elapsed, 3), games_per_s=round(n_games / elapsed, 1),
                moves_per_s=round(moves / elapsed, 1), searches_per_s=round(searches / elapsed, 1),
                ms_per_call=round(1000 * elapsed / calls, 2), wins=wins, draws=draws, losses=losses)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--seconds", type=float, default=1.0)
    ap.add_argument("--workloads", default="tictactoe,connect4")
    args = ap.parse_args()
    name, power = gpu_info()
    for game in args.workloads.split(","):
        games, N = WORKLOADS[game]
        for muzero_player in (0, 1):
            line = run(game, games, N, muzero_player, args.seconds)
            line.update(gpu=name, power_limit=power)
            print(json.dumps(line), flush=True)


if __name__ == "__main__":
    main()
