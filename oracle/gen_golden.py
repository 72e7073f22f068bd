"""ORACLE support: generate the golden fixtures under tests/golden/ FROM THE REFERENCE ITSELF.

Run here (``python -m oracle.gen_golden``), where /root/reference exists; the GPU box only
ever sees the committed outputs.  The reference is imported unmodified (stub ray/gym, see
``oracle/refload.py``) and driven through its own public entry points:

* ``models.MuZeroNetwork(cfg).initial_inference / recurrent_inference``   (net_*.npz)
* ``models.support_to_scalar``, ``MCTS.ucb_score``, ``MinMaxStats``,
  ``SelfPlay.select_action``, ``GameHistory.get_stacked_observations``      (kat.json)
* ``MCTS(cfg).run(...)`` with per-simulation traces captured by wrapping
  ``Node.expand`` / ``MCTS.backpropagate`` / ``numpy.random.*``            (mcts_*.json)
* ``SelfPlay.play_game`` on the reference's own TicTacToe / Connect4 envs  (play_*.json)
* the reference environments themselves on random playouts                 (env_*.json)

It also asserts, at generation time, that this repo's ``weights_spec`` / configs / board
environments agree with the reference's (keys, shapes, attribute values, trajectories).
Weights are ``muzero_general_b200.netspec.synthetic_weights(spec, seed)`` loaded through
the reference's ``set_weights`` - reproducible without the reference - plus the shipped
CartPole checkpoint (stored in the fixture because it cannot be regenerated).
"""
import json
import math
import os
import sys

import numpy
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from muzero_general_b200.netspec import netspec_from_config, synthetic_weights, weights_spec  # noqa: E402
from oracle.refload import REFERENCE_ROOT, load_reference, load_reference_game  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")
torch.set_num_threads(1)


def to_torch_sd(npw):
    return {k: torch.from_numpy(numpy.asarray(v).copy()) for k, v in npw.items()}


def f64list(x):
    return [float(v) for v in x]


# ------------------------------------------------------------------------------- tracing
class Tracer:
    """Wraps reference functions to record what one MCTS.run did, without changing it."""

    def __init__(self, sp):
        self.sp = sp
        self.reset()

    def reset(self):
        self.expands = []      # (reward, priors)
        self.backups = []      # (path_len, value, to_play)
        self.picks = []        # actions chosen by select_child, in call order
        self.dirichlet = []
        self.choices = []      # (n_candidates, picked_index or None for p-sampling)

    def __enter__(self):
        sp, tr = self.sp, self
        self._expand, self._bp, self._sel = sp.Node.expand, sp.MCTS.backpropagate, sp.MCTS.select_child
        self._dir, self._choice = numpy.random.dirichlet, numpy.random.choice

        def expand(node, actions, to_play, reward, policy_logits, hidden_state):
            tr._expand(node, actions, to_play, reward, policy_logits, hidden_state)
            tr.expands.append((float(reward), [float(node.children[a].prior) for a in actions]))

        def backprop(mcts, search_path, value, to_play, mm):
            tr.backups.append((len(search_path), float(value), int(to_play)))
            return tr._bp(mcts, search_path, value, to_play, mm)

        def select(mcts, node, mm):
            a, child = tr._sel(mcts, node, mm)
            tr.picks.append(int(a))
            return a, child

        def dirichlet(alpha, *a, **k):
            out = tr._dir(alpha, *a, **k)
            tr.dirichlet.append(f64list(out))
            return out

        def choice(a, *args, **kw):
            out = tr._choice(a, *args, **kw)
            cand = list(a) if hasattr(a, "__len__") else list(range(a))
            tr.choices.append((len(cand), cand.index(out) if kw.get("p") is None and len(args) < 3 else None))
            return out

        sp.Node.expand, sp.MCTS.backpropagate, sp.MCTS.select_child = expand, backprop, select
        numpy.random.dirichlet, numpy.random.choice = dirichlet, choice
        return self

    def __exit__(self, *exc):
        sp = self.sp
        sp.Node.expand, sp.MCTS.backpropagate, sp.MCTS.select_child = self._expand, self._bp, self._sel
        numpy.random.dirichlet, numpy.random.choice = self._dir, self._choice


def run_traced_search(sp, cfg, model, obs, legal, to_play, add_noise, seed):
    numpy.random.seed(seed)
    with Tracer(sp) as tr, torch.no_grad():
        root, info = sp.MCTS(cfg).run(model, obs, legal, to_play, add_noise)
    # split the flat pick list into per-simulation paths using the backup path lengths
    sims, k = [], 0
    for i, (plen, value, tp) in enumerate(tr.backups):
        depth = plen - 1
        reward, priors = tr.expands[i + 1]
        sims.append(dict(actions=tr.picks[k:k + depth], value=value, reward=reward, priors=priors,
                         leaf_to_play=tp))
        k += depth
    assert k == len(tr.picks)
    first = None
    later_ties = 0
    for j, (n, idx) in enumerate(tr.choices):
        if j == 0:
            first = idx
        elif n > 1:
            later_ties += 1
    kids = list(root.children.keys())
    return dict(
        seed=seed, obs=numpy.asarray(obs).astype(numpy.float64).ravel().tolist(),
        obs_shape=list(numpy.asarray(obs).shape), legal=[int(a) for a in legal], to_play=int(to_play),
        add_noise=bool(add_noise), num_simulations=int(cfg.num_simulations),
        root_reward=tr.expands[0][0], root_priors_raw=tr.expands[0][1],
        noise=tr.dirichlet[0] if tr.dirichlet else None,
        first_index=first, later_ties=later_ties,
        root_priors=[float(root.children[a].prior) for a in kids],
        root_actions=[int(a) for a in kids],
        root_visits=[int(root.children[a].visit_count) for a in kids],
        root_child_value_sums=[float(root.children[a].value_sum) for a in kids],
        root_value=float(root.value()), root_value_sum=float(root.value_sum),
        max_tree_depth=int(info["max_tree_depth"]),
        root_predicted_value=float(info["root_predicted_value"]),
        sims=sims,
    )


# ------------------------------------------------------------------------------- sections
def check_config_and_spec(models, name, ref_cfg, my_cfg):
    skip = {"results_path", "train_on_gpu"}
    for k, v in vars(ref_cfg).items():
        if k in skip:
            continue
        mine = getattr(my_cfg, k)
        assert mine == v, f"{name}: config attribute {k}: reference {v!r} != ours {mine!r}"
    for steps in (0, 1, ref_cfg.training_steps * 0.5, ref_cfg.training_steps * 0.74,
                  ref_cfg.training_steps * 0.75, ref_cfg.training_steps, 5e5, 7.5e5 - 1, 7.5e5):
        assert ref_cfg.visit_softmax_temperature_fn(steps) == my_cfg.visit_softmax_temperature_fn(steps), \
            (name, steps)
    spec = netspec_from_config(my_cfg)
    ref_sd = models.MuZeroNetwork(ref_cfg).get_weights()
    ours = weights_spec(spec)
    assert [k for k, _ in ours] == list(ref_sd.keys()), f"{name}: state_dict key order differs"
    for k, shape in ours:
        assert tuple(ref_sd[k].shape) == tuple(shape), (name, k, shape, ref_sd[k].shape)
    return spec


def gen_kat(sp, models, cart_cfg):
    kat = {}
    rs = numpy.random.RandomState(123)
    logits = (3 * rs.standard_normal((6, 21))).astype(numpy.float32)
    logits[0] = 0; logits[0, 12] = 5; logits[0, 3] = 2
    centre = torch.log(torch.zeros(1, 21).scatter(1, torch.tensor([[10]]).long(), 1.0))
    with numpy.errstate(divide="ignore"):
        out = models.support_to_scalar(torch.from_numpy(logits), 10)[:, 0]
    kat["support_to_scalar"] = dict(logits=logits.tolist(), out=f64list(out),
                                    centre_out=float(models.support_to_scalar(centre, 10).item()),
                                    centre_sign_negative=bool(math.copysign(1, models.support_to_scalar(centre, 10).item()) < 0))
    # ucb_score
    cases = []
    for players in (1, 2):
        cart_cfg.players = list(range(players))
        m = sp.MCTS(cart_cfg)
        for (pn, prior, cn, vsum, rew, lo, hi) in [
            (7, 0.3, 2, 1.5, 1.0, 0.5, 3.0), (0, 0.5, 0, 0, 0, None, None), (1, 0.25, 0, 0, 0, 0.1, 0.1),
            (49, 0.61234, 17, -3.25, 0.5, -1.0, 2.0), (200, 1e-3, 1, 0.75, 10.0, 0.0, 10.0),
        ]:
            parent, child, mm = sp.Node(0), sp.Node(prior), sp.MinMaxStats()
            parent.visit_count = pn
            child.visit_count, child.value_sum, child.reward = cn, vsum, rew
            if lo is not None:
                mm.update(lo); mm.update(hi)
            cases.append(dict(players=players, parent_visits=pn, prior=prior, visits=cn, value_sum=vsum,
                              reward=rew, lo=lo, hi=hi, discount=cart_cfg.discount,
                              pb_c_base=cart_cfg.pb_c_base, pb_c_init=cart_cfg.pb_c_init,
                              score=float(m.ucb_score(parent, child, mm))))
    cart_cfg.players = [0]
    kat["ucb_score"] = cases
    # select_action
    sel = []
    for seed, counts, temp in [(0, [2, 23], 1.0), (1, [7, 43], 0.5), (2, [6, 0, 0, 0, 18, 0, 0, 0, 1], 1.0),
                               (3, [5, 5, 5], 0), (4, [1, 2, 3, 4], float("inf")), (5, [10, 30, 10], 0.25)]:
        node = sp.Node(0)
        for a, c in enumerate(counts):
            node.children[a * 2 + 1] = sp.Node(0.1)
            node.children[a * 2 + 1].visit_count = c
        numpy.random.seed(seed)
        act = sp.SelfPlay.select_action(node, temp)
        sel.append(dict(seed=seed, actions=[a * 2 + 1 for a in range(len(counts))], counts=counts,
                        temperature=("inf" if temp == float("inf") else temp), action=int(act)))
    kat["select_action"] = sel
    # stacked observations
    gh = sp.GameHistory()
    rs = numpy.random.RandomState(5)
    for t in range(4):
        gh.observation_history.append(rs.randint(0, 3, size=(2, 2, 3)).astype("int32"))
        gh.action_history.append(int(rs.randint(0, 5)))
    stk = []
    for index, s in [(-1, 2), (0, 2), (1, 3), (3, 0)]:
        o = gh.get_stacked_observations(index, s, 5)
        stk.append(dict(index=index, stacked=s, shape=list(o.shape), dtype=str(o.dtype), data=o.ravel().tolist()))
    kat["stacked_observations"] = dict(
        observations=[o.tolist() for o in gh.observation_history], actions=gh.action_history, A=5, cases=stk)
    # store_search_statistics
    root = sp.Node(0)
    root.visit_count, root.value_sum = 25, 3.5
    for a, c in [(0, 6), (4, 18), (8, 1)]:
        root.children[a] = sp.Node(0.1)
        root.children[a].visit_count = c
    gh2 = sp.GameHistory()
    gh2.store_search_statistics(root, list(range(9)))
    gh2.store_search_statistics(None, list(range(9)))
    kat["search_statistics"] = dict(child_visits=gh2.child_visits, root_values=gh2.root_values)
    return kat


def gen_net(models, name, ref_cfg, spec, weights, batch, seed):
    net = models.MuZeroNetwork(ref_cfg)
    net.set_weights(to_torch_sd(weights))
    net.eval()
    rs = numpy.random.RandomState(seed)
    if name in ("tictactoe", "connect4", "gomoku"):
        obs = rs.randint(0, 2, size=(batch, spec.in_channels) + spec.obs_shape[1:]).astype(numpy.float32)
        obs[:, -1] = rs.choice([-1.0, 1.0], size=(batch, 1, 1))
    else:
        obs = rs.random_sample((batch, spec.in_channels) + spec.obs_shape[1:]).astype(numpy.float32)
        if name == "cartpole":
            obs = (obs - 0.5) * 0.4
    act = rs.randint(0, spec.action_space, size=(batch, 1)).astype(numpy.int64)
    with torch.no_grad():
        v0, r0, p0, h0 = net.initial_inference(torch.from_numpy(obs))
        v1, r1, p1, h1 = net.recurrent_inference(h0, torch.from_numpy(act))
        v2, r2, p2, h2 = net.recurrent_inference(h1, torch.from_numpy((act + 1) % spec.action_space))
        s = lambda t: models.support_to_scalar(t, ref_cfg.support_size).numpy()[:, 0]
        out = dict(obs=obs, action=act,
                   init_value=v0.numpy(), init_policy=p0.numpy(), init_hidden=h0.numpy(),
                   init_value_scalar=s(v0), init_reward_scalar=s(r0),
                   rec_value=v1.numpy(), rec_reward=r1.numpy(), rec_policy=p1.numpy(), rec_hidden=h1.numpy(),
                   rec_value_scalar=s(v1), rec_reward_scalar=s(r1),
                   rec2_value=v2.numpy(), rec2_reward=r2.numpy(), rec2_policy=p2.numpy(), rec2_hidden=h2.numpy())
    numpy.savez_compressed(os.path.join(OUT, f"net_{name}.npz"), **out)
    return net


def board_obs(game_mod, moves):
    g = game_mod.Game(0)
    obs = g.reset()
    for a in moves:
        obs, _, _ = g.step(a)
    return obs, g.legal_actions(), g.to_play()


def gen_env_fixture(game_mod, my_mod, name, n_games, seed):
    """Random playouts on the reference env; asserts our env agrees step by step."""
    rs = numpy.random.RandomState(seed)
    games = []
    for g in range(n_games):
        ref, mine = game_mod.Game(g), my_mod.Game(g)
        o_r, o_m = ref.reset(), mine.reset()
        assert numpy.array_equal(numpy.asarray(o_r), o_m) and numpy.asarray(o_r).dtype == o_m.dtype, name
        steps, done = [], False
        while not done:
            legal = ref.legal_actions()
            assert legal == mine.legal_actions() and ref.to_play() == mine.to_play()
            a = int(legal[rs.randint(len(legal))])
            o_r, r_r, done = ref.step(a)
            o_m, r_m, d_m = mine.step(a)
            assert numpy.array_equal(numpy.asarray(o_r), o_m) and r_r == r_m and done == d_m, (name, g, a)
            steps.append(dict(action=a, reward=int(r_r), done=bool(done), to_play=int(ref.to_play()),
                              legal=[int(x) for x in ref.legal_actions()],
                              obs=numpy.asarray(o_r).astype(numpy.int8).ravel().tolist()))
        games.append(steps)
    return dict(name=name, obs_dtype=str(numpy.asarray(o_r).dtype), games=games)


def gen_play(sp, game_mod, ref_cfg, weights, seed, temperature):
    ck = {"weights": to_torch_sd(weights)}
    worker = sp.SelfPlay(ck, game_mod.Game, ref_cfg, seed)
    with Tracer(sp) as tr:
        gh = worker.play_game(temperature, ref_cfg.temperature_threshold, False, "self", 0)
    # per-move draws in consumption order: dirichlet, first tie index, [later ties], action sample
    return dict(
        seed=seed, temperature=temperature, num_simulations=int(ref_cfg.num_simulations),
        action_history=[int(a) for a in gh.action_history],
        reward_history=[float(r) for r in gh.reward_history],
        to_play_history=[int(t) for t in gh.to_play_history],
        child_visits=[f64list(c) for c in gh.child_visits],
        root_values=f64list(gh.root_values),
        observation_history=[numpy.asarray(o).astype(numpy.float64).ravel().tolist() for o in gh.observation_history],
        dirichlet=tr.dirichlet, choices=[[n, idx] for n, idx in tr.choices],
    )


def main():
    os.makedirs(OUT, exist_ok=True)
    sp, models, replay_buffer, trainer = load_reference()
    import muzero_general_b200.games as mygames

    manifest = {"reference_root": REFERENCE_ROOT, "torch": torch.__version__, "numpy": numpy.__version__}
    specs, ref_cfgs, ref_games = {}, {}, {}
    for name in ("cartpole", "tictactoe", "connect4", "breakout"):
        ref_games[name] = load_reference_game(name)
        ref_cfgs[name] = ref_games[name].MuZeroConfig()
        my_cfg = mygames.load_game_module(name).MuZeroConfig()
        specs[name] = check_config_and_spec(models, name, ref_cfgs[name], my_cfg)
    print("configs + weights_spec agree with the reference for", list(specs))

    json.dump(gen_kat(sp, models, load_reference_game("cartpole").MuZeroConfig()),
              open(os.path.join(OUT, "kat.json"), "w"))

    # ---- environments
    for name, n in (("tictactoe", 24), ("connect4", 12)):
        fx = gen_env_fixture(ref_games[name], mygames.load_game_module(name), name, n, seed=11)
        json.dump(fx, open(os.path.join(OUT, f"env_{name}.json"), "w"))
    print("board environments agree with the reference")

    # ---- networks + searches
    nets = {}
    for name, batch in (("cartpole", 8), ("tictactoe", 8), ("connect4", 4), ("breakout", 2)):
        w = synthetic_weights(specs[name], seed=0)
        nets[name] = gen_net(models, name, ref_cfgs[name], specs[name], w, batch, seed=3)
    print("network fixtures written")

    searches = {}
    # CartPole, synthetic weights, N = 25 and 50, noise on/off
    cfg = ref_cfgs["cartpole"]
    obs = numpy.array([[[0.01, -0.02, 0.03, 0.04]]], dtype=numpy.float32)
    runs = []
    for n_sim, noise, seed in ((25, True, 0), (50, True, 0), (50, False, 1), (50, True, 7)):
        cfg.num_simulations = n_sim
        runs.append(run_traced_search(sp, cfg, nets["cartpole"], obs, [0, 1], 0, noise, seed))
    searches["cartpole_synth"] = runs
    # CartPole, the shipped checkpoint
    ck = torch.load(os.path.join(REFERENCE_ROOT, "results", "cartpole", "model.checkpoint"),
                    map_location="cpu", weights_only=False)
    pre = models.MuZeroNetwork(cfg)
    pre.set_weights(ck["weights"])
    pre.eval()
    numpy.savez_compressed(os.path.join(OUT, "weights_cartpole_pretrained.npz"),
                           **{k: v.numpy() for k, v in ck["weights"].items()})
    runs = []
    for n_sim, noise, seed in ((25, True, 0), (50, True, 0), (50, False, 0)):
        cfg.num_simulations = n_sim
        runs.append(run_traced_search(sp, cfg, pre, obs, [0, 1], 0, noise, seed))
    searches["cartpole_pretrained"] = runs
    cfg.num_simulations = 50

    # TicTacToe: opening, mid-game (restricted legal set, player 1 to move)
    cfg = ref_cfgs["tictactoe"]
    runs = []
    for moves, n_sim, seed in (((), 25, 0), ((4, 0, 8), 50, 1), ((0, 1, 2, 4), 50, 2)):
        cfg.num_simulations = n_sim
        o, legal, tp = board_obs(ref_games["tictactoe"], moves)
        runs.append(run_traced_search(sp, cfg, nets["tictactoe"], o, legal, tp, True, seed))
    searches["tictactoe"] = runs
    cfg.num_simulations = 25

    cfg = ref_cfgs["connect4"]
    runs = []
    for moves, n_sim, seed in (((), 40, 0), ((3, 3, 2, 4, 3, 3, 3, 3), 60, 1)):
        cfg.num_simulations = n_sim
        o, legal, tp = board_obs(ref_games["connect4"], moves)
        runs.append(run_traced_search(sp, cfg, nets["connect4"], o, legal, tp, True, seed))
    searches["connect4"] = runs
    cfg.num_simulations = 200

    cfg = ref_cfgs["breakout"]
    cfg.num_simulations = 12
    o = numpy.random.RandomState(9).random_sample((3, 96, 96)).astype(numpy.float32)
    searches["breakout"] = [run_traced_search(sp, cfg, nets["breakout"], o, [0, 1, 2, 3], 0, True, 4)]
    cfg.num_simulations = 30
    for k, v in searches.items():
        json.dump(v, open(os.path.join(OUT, f"mcts_{k}.json"), "w"))
    print("search fixtures written")

    # ---- whole games on the reference's own environments
    plays = {}
    cfg = ref_cfgs["tictactoe"]
    plays["tictactoe"] = [gen_play(sp, ref_games["tictactoe"], cfg, synthetic_weights(specs["tictactoe"], 0), s, t)
                          for s, t in ((0, 0), (1, 1.0), (2, 0.5))]
    cfg = ref_cfgs["connect4"]
    cfg.num_simulations = 30
    plays["connect4"] = [gen_play(sp, ref_games["connect4"], cfg, synthetic_weights(specs["connect4"], 0), 0, 1.0)]
    cfg.num_simulations = 200
    json.dump(plays, open(os.path.join(OUT, "play.json"), "w"))
    json.dump(manifest, open(os.path.join(OUT, "MANIFEST.json"), "w"), indent=1)
    main_round2()
    print("done ->", OUT)


def layer_extrema(models, net, obs, act):
    """Largest |activation| after every conv/BN/ReLU stage of the three towers (forward hooks on the reference)."""
    peaks = {}

    def hook(name):
        def fn(mod, inp, out):
            peaks[name] = max(peaks.get(name, 0.0), float(out.detach().abs().max()))
        return fn

    handles = [m.register_forward_hook(hook(n)) for n, m in net.named_modules()
               if isinstance(m, (torch.nn.BatchNorm2d, models.ResidualBlock))]
    with torch.no_grad():
        _, _, _, h = net.initial_inference(torch.from_numpy(obs))
        net.recurrent_inference(h, torch.from_numpy(act))
    for hd in handles:
        hd.remove()
    return peaks


def main_round2():
    """Round-2 fixtures: the BASELINE closed-loop configs (Connect4 N=200, Breakout N=50), a batch-64 Connect4
    network fixture, and network fixtures on STRESS weights (activations up to ~1e4, beyond the fp16 range, and
    down to ~1e-5) for the tensor-core towers' range guard.  Existing fixtures are untouched."""
    from muzero_general_b200.netspec import stress_weights
    sp, models, replay_buffer, trainer = load_reference()
    specs, ref_cfgs, ref_games = {}, {}, {}
    for name in ("connect4", "breakout"):
        ref_games[name] = load_reference_game(name)
        ref_cfgs[name] = ref_games[name].MuZeroConfig()
        specs[name] = netspec_from_config(ref_cfgs[name])

    def ref_net(name, weights):
        net = models.MuZeroNetwork(ref_cfgs[name])
        net.set_weights(to_torch_sd(weights))
        net.eval()
        return net

    # ---- closed loop at the BASELINE simulation counts
    cfg = ref_cfgs["connect4"]
    net = ref_net("connect4", synthetic_weights(specs["connect4"], 0))
    runs = []
    for moves, seed in (((), 0), ((3, 3, 2, 4, 3, 3, 3, 3), 1), ((0, 6, 1, 5, 2), 2)):
        cfg.num_simulations = 200
        o, legal, tp = board_obs(ref_games["connect4"], moves)
        runs.append(run_traced_search(sp, cfg, net, o, legal, tp, True, seed))
    json.dump(runs, open(os.path.join(OUT, "mcts_connect4_n200.json"), "w"))
    cfg = ref_cfgs["breakout"]
    net = ref_net("breakout", synthetic_weights(specs["breakout"], 0))
    cfg.num_simulations = 50
    runs = []
    for obs_seed, seed in ((19, 5),):
        o = numpy.random.RandomState(obs_seed).random_sample((3, 96, 96)).astype(numpy.float32)
        runs.append(run_traced_search(sp, cfg, net, o, [0, 1, 2, 3], 0, True, seed))
    cfg.num_simulations = 30
    json.dump(runs, open(os.path.join(OUT, "mcts_breakout_n50.json"), "w"))
    print("BASELINE-size closed-loop fixtures written")

    # ---- the wide-action-space game: environment trajectories and a network + search fixture for games/gomoku.py
    import muzero_general_b200.games as mygames2
    go_ref = load_reference_game("gomoku")
    fx = gen_env_fixture(go_ref, mygames2.load_game_module("gomoku"), "gomoku", 6, seed=13)
    json.dump(fx, open(os.path.join(OUT, "env_gomoku.json"), "w"))
    go_cfg = go_ref.MuZeroConfig()
    go_spec = check_config_and_spec(models, "gomoku", go_cfg, mygames2.load_game_module("gomoku").MuZeroConfig())
    go_net = gen_net(models, "gomoku", go_cfg, go_spec, synthetic_weights(go_spec, 0), 3, seed=5)
    runs = []
    for moves, n_sim, seed in (((), 60, 0), ((60, 61, 49, 71, 38), 90, 1)):
        go_cfg.num_simulations = n_sim
        o, legal, tp = board_obs(go_ref, moves)
        runs.append(run_traced_search(sp, go_cfg, go_net, o, legal, tp, True, seed))
    go_cfg.num_simulations = 400
    json.dump(runs, open(os.path.join(OUT, "mcts_gomoku.json"), "w"))
    print("gomoku fixtures written")

    # ---- hard-coded opponents (expert_agent): reference choice at every position of random playouts
    experts = {}
    for gname in ("tictactoe", "connect4"):
        gm = load_reference_game(gname)
        rs = numpy.random.RandomState(23)
        cases = []
        for g in range(40):
            ref = gm.Game(g)
            ref.reset()
            moves, done = [], False
            while not done:
                seed = len(cases)
                numpy.random.seed(seed)
                cases.append(dict(moves=list(moves), seed=seed, action=int(ref.expert_agent())))
                legal = ref.legal_actions()
                # mostly random moves, sometimes the expert's own, so that threats of both colours show up
                a = cases[-1]["action"] if rs.uniform() < 0.3 else int(legal[rs.randint(len(legal))])
                _, _, done = ref.step(a)
                moves.append(a)
        experts[gname] = cases
    json.dump(experts, open(os.path.join(OUT, "expert.json"), "w"))
    print("expert fixtures:", {k: len(v) for k, v in experts.items()})

    # ---- override_root_with (self_play.py:275-277): (a) subtree reuse - the most visited child of a finished search
    # becomes the root of a second search; (b) diagnose_model.py:54-69 - a hand-expanded, unvisited root
    over = {}
    for gname, moves in (("tictactoe", (4, 0)), ("cartpole", None)):
        gm = load_reference_game(gname)
        rcfg = gm.MuZeroConfig()
        rcfg.num_simulations = 25
        rspec = netspec_from_config(rcfg)
        wts = synthetic_weights(rspec, 0)
        rnet = models.MuZeroNetwork(rcfg); rnet.set_weights(to_torch_sd(wts)); rnet.eval()
        if moves is None:
            o, legal, tp = numpy.array([[[0.01, -0.02, 0.03, 0.04]]], dtype=numpy.float32), [0, 1], 0
        else:
            o, legal, tp = board_obs(gm, moves)
        first = run_traced_search(sp, rcfg, rnet, o, legal, tp, True, 0)
        cases = []
        for kind in ("subtree", "fresh"):
            numpy.random.seed(0)
            with torch.no_grad():
                root, _ = sp.MCTS(rcfg).run(rnet, o, legal, tp, True)
                action = int(sp.SelfPlay.select_action(root, 0))
                ntp = rcfg.players[tp + 1] if tp + 1 < len(rcfg.players) else rcfg.players[0]
                if kind == "subtree":
                    node = root.children[action]
                else:
                    value, reward, policy_logits, hidden_state = rnet.recurrent_inference(root.hidden_state, torch.tensor([[action]]))
                    reward = models.support_to_scalar(reward, rcfg.support_size).item()
                    node = sp.Node(0)
                    node.expand(rcfg.action_space, ntp, reward, policy_logits, hidden_state)
                pre_visits = int(node.visit_count)
                with Tracer(sp) as tr:
                    root2, info2 = sp.MCTS(rcfg).run(rnet, None, rcfg.action_space, ntp, True, node)
            kids = list(root2.children.keys())
            cases.append(dict(kind=kind, action=action, to_play=int(ntp), pre_visits=pre_visits,
                              noise=tr.dirichlet[0], choices=[[n, i] for n, i in tr.choices],
                              root_actions=[int(a) for a in kids],
                              root_visits=[int(root2.children[a].visit_count) for a in kids],
                              root_child_value_sums=[float(root2.children[a].value_sum) for a in kids],
                              root_priors=[float(root2.children[a].prior) for a in kids],
                              root_visit_count=int(root2.visit_count), root_value=float(root2.value()),
                              max_tree_depth=int(info2["max_tree_depth"]),
                              root_predicted_value=info2["root_predicted_value"]))
        over[gname] = dict(first=first, cases=cases)
    json.dump(over, open(os.path.join(OUT, "override_root.json"), "w"))
    print("override_root_with fixtures:", {k: [c["root_visits"] for c in v["cases"]] for k, v in over.items()})

    # ---- the large configuration (games/atari.py: 131 stacked input planes, 16 blocks x 256 channels, 601-bin heads):
    # outputs only - the 9.6 MB observation batch is regenerated from its seed by the tests
    import muzero_general_b200.games as mygames
    at_ref = load_reference_game("atari").MuZeroConfig()
    at_spec = check_config_and_spec(models, "atari", at_ref, mygames.load_game_module("atari").MuZeroConfig())
    at_net = models.MuZeroNetwork(at_ref)
    at_net.set_weights(to_torch_sd(synthetic_weights(at_spec, 0)))
    at_net.eval()
    at_obs = numpy.random.RandomState(41).random_sample((2, at_spec.in_channels, 96, 96)).astype(numpy.float32)
    at_act = numpy.array([[1], [3]], dtype=numpy.int64)
    with torch.no_grad():
        v0, r0, p0, h0 = at_net.initial_inference(torch.from_numpy(at_obs))
        v1, r1, p1, h1 = at_net.recurrent_inference(h0, torch.from_numpy(at_act))
        sc = lambda t: models.support_to_scalar(t, at_ref.support_size).numpy()[:, 0]
        numpy.savez_compressed(os.path.join(OUT, "net_atari.npz"), obs_seed=41, action=at_act,
                               init_value=v0.numpy(), init_policy=p0.numpy(), init_hidden=h0.numpy(), init_value_scalar=sc(v0),
                               rec_value=v1.numpy(), rec_reward=r1.numpy(), rec_policy=p1.numpy(), rec_hidden=h1.numpy(),
                               rec_value_scalar=sc(v1), rec_reward_scalar=sc(r1))
    del at_net
    print("large-configuration network fixture written")

    # ---- FC network on the shipped CartPole checkpoint (the round-1 fixture only covered synthetic weights)
    cart_mod = load_reference_game("cartpole")
    cart_cfg = cart_mod.MuZeroConfig()
    cart_spec = netspec_from_config(cart_cfg)
    pre = dict(numpy.load(os.path.join(OUT, "weights_cartpole_pretrained.npz")))
    os.rename(os.path.join(OUT, "net_cartpole.npz"), os.path.join(OUT, "net_cartpole.keep"))
    gen_net(models, "cartpole", cart_cfg, cart_spec, pre, 16, seed=29)
    os.rename(os.path.join(OUT, "net_cartpole.npz"), os.path.join(OUT, "net_cartpole_pretrained.npz"))
    os.rename(os.path.join(OUT, "net_cartpole.keep"), os.path.join(OUT, "net_cartpole.npz"))

    # ---- larger network batches
    name = "connect4"
    w = synthetic_weights(specs[name], seed=0)
    os.rename(os.path.join(OUT, f"net_{name}.npz"), os.path.join(OUT, f"net_{name}.keep"))
    gen_net(models, name, ref_cfgs[name], specs[name], w, 64, seed=13)
    os.rename(os.path.join(OUT, f"net_{name}.npz"), os.path.join(OUT, f"net_{name}_b64.npz"))
    # ---- stress weights
    info = {}
    for mode in ("large", "overflow", "tiny"):
        w = stress_weights(specs[name], 0, mode)
        net = gen_net(models, name, ref_cfgs[name], specs[name], w, 8, seed=17)
        os.rename(os.path.join(OUT, f"net_{name}.npz"), os.path.join(OUT, f"net_{name}_stress_{mode}.npz"))
        g = dict(numpy.load(os.path.join(OUT, f"net_{name}_stress_{mode}.npz")))
        peaks = layer_extrema(models, net, g["obs"], g["action"])
        info[mode] = dict(max_activation=max(peaks.values()), min_layer_peak=min(peaks.values()))
        print("stress", mode, info[mode])
    os.rename(os.path.join(OUT, f"net_{name}.keep"), os.path.join(OUT, f"net_{name}.npz"))
    json.dump(info, open(os.path.join(OUT, "net_connect4_stress_info.json"), "w"), indent=1)
    print("network fixtures (batch 64, stress weights) written")


def priority_key(name, td, discount, alpha, reanalysed):
    return f"{name}/td{td}/discount{discount}/alpha{alpha}/reanalysed{int(reanalysed)}"


# (game, td_steps, discount, PER_alpha, reanalysed values): one- and two-player games, short and long td horizons
PRIORITY_CASES = [("tictactoe", 20, 1, 0.5, False), ("cartpole", 50, 0.997, 0.5, False),
                  ("cartpole", 7, 0.9, 1.0, True), ("connect4", 3, 1, 0.7, True)]
PRIORITY_LENGTHS = (1, 2, 9, 42, 130)


def main_replay():
    """replay_buffer.json: what the reference's ReplayBuffer computes from game histories.

    * ``priorities``: ``save_game``'s PER priorities and game priority of random histories
      (``tests/helpers.random_history``, RandomState(4), game lengths PRIORITY_LENGTHS per case).
    * ``batch``: ``save_game`` + ``get_batch`` (batch_size 8) over six TicTacToe games played by THIS package's
      ``SelfPlay`` (seed 1, 4 parallel games, 8 simulations, synthetic weights seed 0, the oracle-backed test double
      in place of the GPU engine), each passed through pickle first."""
    import copy
    import pickle
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from fake_engine import FakeSearchEngine
    from helpers import random_history
    from muzero_general_b200 import self_play as mysp
    import muzero_general_b200.games as mygames
    _, _, ref_rb, _ = load_reference()
    ck = {"num_played_games": 0, "num_played_steps": 0}

    priorities = {}
    for name, td, discount, alpha, reanalysed in PRIORITY_CASES:
        cfg = load_reference_game(name).MuZeroConfig()
        cfg.td_steps, cfg.discount, cfg.PER_alpha, cfg.PER = td, discount, alpha, True
        rs = numpy.random.RandomState(4)
        rows = []
        for T in PRIORITY_LENGTHS:
            gh = random_history(rs, cfg, T, len(cfg.players))
            if reanalysed:
                gh.reanalysed_predicted_root_values = rs.standard_normal(T).astype(numpy.float32)
            ref_rb.ReplayBuffer(copy.deepcopy(ck), {}, cfg).save_game(gh)
            assert gh.priorities.dtype == numpy.float32
            rows.append(dict(T=T, priorities=f64list(gh.priorities), game_priority=float(gh.game_priority)))
        priorities[priority_key(name, td, discount, alpha, reanalysed)] = rows

    mod = mygames.load_game_module("tictactoe")
    my_cfg = mod.MuZeroConfig()
    my_cfg.num_parallel_games, my_cfg.num_simulations = 4, 8
    mysp.SearchEngine = FakeSearchEngine
    worker = mysp.SelfPlay({"weights": synthetic_weights(netspec_from_config(my_cfg), 0)}, mod.Game, my_cfg, 1)
    games = worker.play_games(6, 1.0)
    cfg = load_reference_game("tictactoe").MuZeroConfig()
    cfg.num_simulations, cfg.batch_size, cfg.train_on_gpu = 8, 8, False
    buf = ref_rb.ReplayBuffer(dict(ck, weights=None), {}, cfg)
    for gh in games:
        buf.save_game(pickle.loads(pickle.dumps(gh)))
    index_batch, (obs_b, act_b, val_b, rew_b, pol_b, _, _) = buf.get_batch()
    batch = dict(num_games=len(games), index=[[int(g), int(p)] for g, p in index_batch],
                 priorities=[f64list(buf.buffer[g].priorities) for g in range(len(games))],
                 game_priority=[float(buf.buffer[g].game_priority) for g in range(len(games))],
                 observation=[numpy.asarray(o, dtype=numpy.float64).ravel().tolist() for o in obs_b],
                 action=[[int(a) for a in r] for r in act_b], value=[f64list(r) for r in val_b],
                 reward=[f64list(r) for r in rew_b], policy=[[f64list(p) for p in r] for r in pol_b])
    json.dump(dict(priorities=priorities, batch=batch), open(os.path.join(OUT, "replay_buffer.json"), "w"))
    print("replay buffer fixtures written")


if __name__ == "__main__":
    if "--round2" in sys.argv:
        main_round2()
    elif "--replay" in sys.argv:
        main_replay()
    else:
        main()
