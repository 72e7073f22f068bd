"""Where the fused FC search kernel's time goes: tree work against network work, at the headline shape.

    python scripts/fc_search_split.py [--games 4096] [--sims 50] [--repeats 20]

Same inputs as bench.py's cartpole_b4096_n50 (synthetic weights seed 0, first batch of RandomState(100): observations
U(+-0.05) and Dirichlet root noise, game ids 0..B-1).  Times, as CUDA-event device time of the search
(SearchOutput.device_ms, the median of --repeats searches):
  full     the whole search: root inference, N x {select, network, expand, backup}
  teacher  the same search with the network replaced by its own traced outputs (teacher mode): the identical tree with
           identical paths, and no network evaluation
The difference is the network's share.  Caveat: the teacher kernel keeps no weights and no hidden states in shared memory
and runs at a different occupancy; at 4096 games both launches are a single wave, so per-warp chain length is what both
times measure.  Each split is taken with MZ_FC_LOOKAHEAD=0 (one tree level per selection round) and =1 (several levels
per round, the default for |A| <= 2); one JSON line per setting, with the GPU's name and power limit read in the same run.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def gpu_info():
    out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True, check=True).stdout.strip()
    name, power = (x.strip() for x in out.split(",", 1))
    return name, power


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--games", type=int, default=4096)
    ap.add_argument("--sims", type=int, default=50)
    ap.add_argument("--repeats", type=int, default=20)
    args = ap.parse_args()
    import numpy
    from muzero_general_b200.engine import SearchEngine
    from muzero_general_b200.games import load_game_module
    from muzero_general_b200.netspec import netspec_from_config, synthetic_weights

    name, power = gpu_info()
    cfg = load_game_module("cartpole").MuZeroConfig()
    spec = netspec_from_config(cfg)
    B, N, A = args.games, args.sims, spec.action_space
    rs = numpy.random.RandomState(100)
    obs = [rs.uniform(-0.05, 0.05, size=(B, 4)).astype(numpy.float32) for _ in range(4)][0]
    noise = [rs.dirichlet([cfg.root_dirichlet_alpha] * A, size=B) for _ in range(4)][0]
    gid = numpy.arange(B, dtype=numpy.int64)
    eng = SearchEngine(cfg, max_games=B, num_simulations=N, seed=cfg.seed)
    eng.load_weights(synthetic_weights(spec, 0))

    def median_ms(fn):
        fn()                                       # warm-up
        return statistics.median(fn().device_ms for _ in range(args.repeats))

    for la in ("0", "1"):
        os.environ["MZ_FC_LOOKAHEAD"] = la
        search = lambda **kw: eng.search(obs=obs, add_exploration_noise=True, noise=noise, game_id=gid, **kw)
        full = median_ms(search)
        traced = search(trace=True)
        tr = traced.trace
        teacher = dict(root_value=traced.root_predicted_value, root_reward=tr["root_reward"],
                       root_priors=tr["root_priors_raw"], value=tr["value"], reward=tr["reward"], priors=tr["priors"])
        legal = numpy.ones((B, A), numpy.uint8)
        replay = lambda: eng.search(legal_mask=legal, add_exploration_noise=True, noise=noise, game_id=gid,
                                    teacher=teacher, n_games=B)
        same = replay()
        assert numpy.array_equal(same.visit_counts, traced.visit_counts) and numpy.array_equal(same.root_value, traced.root_value)
        tree = median_ms(replay)
        depth = tr["depth"]
        print(json.dumps(dict(lookahead=int(la), games=B, num_simulations=N, repeats=args.repeats,
                              full_ms=round(full, 4), teacher_ms=round(tree, 4), network_ms=round(full - tree, 4),
                              tree_share=round(tree / full, 3), mean_depth=round(float(depth.mean()), 3),
                              max_depth=int(depth.max()), gpu=name, power_limit=power)), flush=True)
    eng.close()


if __name__ == "__main__":
    main()
