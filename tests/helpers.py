"""Shared test helpers (also used by oracle/gen_golden.py): teacher tables from golden traces, oracle replays,
random game histories."""
import numpy

from oracle import mcts as om
from oracle import philox


def teacher_from_cases(cases, A, N):
    """Stack golden search cases (same N) into the arrays mz_search's teacher mode takes."""
    n = len(cases)
    t = dict(root_value=numpy.zeros(n, numpy.float32), root_reward=numpy.zeros(n, numpy.float32),
             root_priors=numpy.zeros((n, A), numpy.float32), value=numpy.zeros((n, N), numpy.float32),
             reward=numpy.zeros((n, N), numpy.float32), priors=numpy.zeros((n, N, A), numpy.float32))
    legal = numpy.zeros((n, A), numpy.uint8)
    noise = numpy.zeros((n, A), numpy.float64)
    first = numpy.full(n, -1, numpy.int32)
    to_play = numpy.zeros(n, numpy.int32)
    for i, c in enumerate(cases):
        assert c["num_simulations"] == N
        t["root_value"][i] = c["root_predicted_value"]
        t["root_reward"][i] = c["root_reward"]
        for k, a in enumerate(c["legal"]):
            t["root_priors"][i, a] = c["root_priors_raw"][k]
            legal[i, a] = 1
            if c["noise"] is not None:
                noise[i, a] = c["noise"][k]
        for s, sim in enumerate(c["sims"]):
            t["value"][i, s] = sim["value"]
            t["reward"][i, s] = sim["reward"]
            t["priors"][i, s] = sim["priors"]
        if c["first_index"] is not None:
            first[i] = c["first_index"]
        to_play[i] = c["to_play"]
    return t, legal, noise, first, to_play


def paths_from_trace(trace, i, N):
    return [[int(a) for a in trace["actions"][i, s, :trace["depth"][i, s]]] for s in range(N)]


def oracle_replay(params, legal, to_play, root, sims, noise, first_index, seed=0, game=0, move=0):
    """Run the oracle tree on a table of per-simulation outputs with the device's tie rule."""
    ev = om.TableEvaluator(root, sims)
    draws = om.InjectedDraws(
        noise, first_index,
        tie_fn=lambda n_tied, ctx: philox.tie_index(seed, game, move, ctx[0], ctx[1], n_tied))
    res = om.TreeSearch(params).run(ev, None, legal, to_play, noise is not None, draws)
    return res, draws


def random_history(rs, cfg, T, players):
    """A GameHistory of T random moves (random observations, rewards, visit distributions and root values)."""
    from muzero_general_b200 import self_play as sp
    gh = sp.GameHistory()
    A = len(cfg.action_space)
    gh.action_history = [0] + [int(a) for a in rs.randint(0, A, T)]
    gh.observation_history = [rs.random_sample(cfg.observation_shape).astype(numpy.float32) for _ in range(T + 1)]
    gh.reward_history = [0] + [float(r) for r in rs.choice([0.0, 1.0, -1.0, 0.5], T)]
    gh.to_play_history = [int(i % players) for i in range(T + 1)] if players > 1 else [0] * (T + 1)
    cv = rs.random_sample((T, A)); gh.child_visits = (cv / cv.sum(1, keepdims=True)).tolist()
    gh.root_values = [float(v) for v in rs.standard_normal(T)]
    return gh


def random_teacher(rs, n, N, A, reward_scale=1.0, legal=None):
    """Synthetic per-simulation network outputs (SURVEY.md 8d): fp32 softmax priors, U(-1,1) values."""
    def soft(x):
        e = numpy.exp(x - x.max(-1, keepdims=True)).astype(numpy.float32)
        return (e / e.sum(-1, keepdims=True)).astype(numpy.float32)
    t = dict(root_value=rs.uniform(-1, 1, n).astype(numpy.float32),
             root_reward=numpy.zeros(n, numpy.float32),
             value=rs.uniform(-1, 1, (n, N)).astype(numpy.float32),
             reward=(reward_scale * rs.uniform(0, 1, (n, N))).astype(numpy.float32),
             priors=soft(rs.standard_normal((n, N, A)).astype(numpy.float32)))
    logits = rs.standard_normal((n, A)).astype(numpy.float32)
    if legal is not None:
        logits = numpy.where(legal > 0, logits, -numpy.inf).astype(numpy.float32)
    t["root_priors"] = soft(logits)
    return t
