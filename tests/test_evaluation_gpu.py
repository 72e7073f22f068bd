"""Evaluation games on the device (mz_selfplay_set_opponent, csrc/selfplay.cu): the device expert against the
reference's recorded expert moves, whole evaluation games against a host replay and the search they wrap,
SelfPlay.play_test_games' batch invariance, the argument checks and the test-mode report."""
import numpy
import pytest

from conftest import golden_json, weights_for
from eval_helpers import TAG_OPPONENT, uniform53
from muzero_general_b200 import _lib
from muzero_general_b200.games import load_game_module
from muzero_general_b200.games._boards import _threat_scan
from muzero_general_b200.netspec import netspec_from_config

pytestmark = pytest.mark.gpu


def _engine(name, B, N, seed=0, **over):
    from muzero_general_b200.engine import SearchEngine
    mod = load_game_module(name)
    cfg = mod.MuZeroConfig()
    for k, v in over.items():
        setattr(cfg, k, v)
    spec = netspec_from_config(cfg)
    eng = SearchEngine(cfg, max_games=B, num_simulations=N, seed=seed)
    eng.load_weights(weights_for(name, spec))
    return mod, cfg, eng


def _eval_loop(name, B, N, opponent, muzero_player, seed=0, **over):
    from muzero_general_b200.engine import DeviceSelfPlayLoop
    mod, cfg, eng = _engine(name, B, N, seed, **over)
    loop = DeviceSelfPlayLoop(eng, name, cfg.max_moves, reward_scale=mod.Game.VECTOR.REWARD_SCALE,
                              opponent=opponent, muzero_player=muzero_player)
    return mod, cfg, eng, loop


@pytest.mark.parametrize("name", ["tictactoe", "connect4"])
def test_device_expert_plays_the_reference_moves(name):
    """Every recorded position of tests/golden/expert.json through mz_debug_opponent_action: with the default draw
    u = (idx + 0.5) / n_legal, idx = the reference's numpy.random.choice after numpy.random.seed(seed), the device
    expert plays the reference's move; the random opponent plays legal[floor(u * n_legal)]."""
    from muzero_general_b200.engine import debug_opponent_action
    mod = load_game_module(name)
    cases = golden_json("expert.json")[name]
    boards, players, uniforms, legal_lists = [], [], [], []
    for c in cases:
        g = mod.Game(0)
        g.reset()
        for a in c["moves"]:
            g.step(a)
        legal = g.legal_actions()
        numpy.random.seed(c["seed"])
        idx = legal.index(int(numpy.random.choice(legal)))
        boards.append(g.env.board[0].copy())
        players.append(int(g.env.player[0]))
        uniforms.append((idx + 0.5) / len(legal))
        legal_lists.append(legal)
    expert = debug_opponent_action(name, "expert", numpy.array(boards), players, uniforms)
    assert expert.tolist() == [c["action"] for c in cases]
    rnd = debug_opponent_action(name, "random", numpy.array(boards), players, uniforms)
    assert rnd.tolist() == [legal[int(u * len(legal))] for legal, u in zip(legal_lists, uniforms)]


@pytest.mark.parametrize("name,B,N", [("tictactoe", 24, 6), ("connect4", 12, 4)])
@pytest.mark.parametrize("opponent", ["expert", "random"])
@pytest.mark.parametrize("muzero_player", [0, 1])
def test_evaluation_games_equal_a_host_replay(name, B, N, opponent, muzero_player, monkeypatch):
    """Every delivered game: moves alternate, MuZero moves exactly when to_play == muzero_player and its rows carry N
    visits, opponent rows NaN / zero visits; opponent moves are the host expert / random pick with the recomputed Philox
    draw; the host environment reproduces observations, rewards and the end; each MuZero row equals SearchEngine.search
    (same seed, device noise) on the recorded observation, its action the first argmax among the legal actions."""
    monkeypatch.setenv("MZ_TC_MODE", "off")
    from muzero_general_b200.engine import parse_staged_games
    seed = 7
    mod, cfg, eng, loop = _eval_loop(name, B, N, opponent, muzero_player, seed=seed)
    games = []
    for _ in range(4):
        loop.moves(cfg.max_moves, 0.0)
        games += parse_staged_games(*loop.drain())
    assert len(games) >= B
    rows = []                               # (game id, move index, observation, legal, to_play, visits, root value)
    for rec in games:
        T, gid = rec["length"], int(rec["game_id"])
        assert 1 <= T <= cfg.max_moves and rec["first_to_play"] == 0
        env = mod.Game(0)
        assert numpy.array_equal(env.reset().astype(numpy.float32).ravel(), rec["obs"][0])
        done = False
        for t in range(T):
            assert not done
            to_play = env.to_play()
            assert to_play == t % 2                                         # moves alternate
            legal = env.legal_actions()
            a = int(rec["action"][t])
            if to_play == muzero_player:
                assert int(rec["visits"][t].sum()) == N and not numpy.isnan(rec["root_value"][t])
                mask = numpy.zeros(len(cfg.action_space), numpy.uint8)
                mask[legal] = 1
                v = rec["visits"][t]
                assert a == max(legal, key=lambda k: (v[k], -k))             # first argmax among the legal actions
                rows.append((gid, t, rec["obs"][t], mask, to_play, v, rec["root_value"][t]))
            else:
                assert not rec["visits"][t].any() and numpy.isnan(rec["root_value"][t])
                u = uniform53(seed, gid, t, 0, TAG_OPPONENT)
                default = legal[min(int(u * len(legal)), len(legal) - 1)]
                if opponent == "expert":
                    board = env.env.board[0].reshape(env.env.H, env.env.W)
                    want = _threat_scan(board, int(env.env.player[0]), env._expert_windows(board), default)
                else:
                    want = default
                assert a == int(want), (gid, t)
            obs, reward, done = env.step(a)
            assert numpy.array_equal(obs.astype(numpy.float32).ravel(), rec["obs"][t + 1])
            assert reward == rec["reward"][t] and env.to_play() == rec["to_play"][t]
        assert done or T == cfg.max_moves
    assert rows
    # the searches, B rows per call like the loop's own calls (padded with the last row)
    _, _, ref = _engine(name, B, N, seed)
    for i in range(0, len(rows), B):
        chunk = rows[i:i + B]
        chunk = chunk + [chunk[-1]] * (B - len(chunk))
        out = ref.search(obs=numpy.stack([r[2] for r in chunk]), legal_mask=numpy.stack([r[3] for r in chunk]),
                         to_play=numpy.array([r[4] for r in chunk], numpy.int32), add_exploration_noise=True,
                         game_id=numpy.array([r[0] for r in chunk], numpy.int64),
                         move_index=numpy.array([r[1] for r in chunk], numpy.int32))
        for j, r in enumerate(rows[i:i + B]):
            assert out.visit_counts[j].tolist() == r[5].tolist(), (r[0], r[1])
            assert out.root_value[j] == r[6]
    eng.close()
    ref.close()


def _worker(name, **over):
    from muzero_general_b200 import self_play as sp
    mod = load_game_module(name)
    cfg = mod.MuZeroConfig()
    cfg.rng_mode, cfg.num_parallel_games, cfg.num_simulations = "philox", 8, 6
    for k, v in over.items():
        setattr(cfg, k, v)
    worker = sp.SelfPlay({"weights": weights_for(name, netspec_from_config(cfg))}, mod.Game, cfg, seed=0)
    assert worker.loop_path == "device"
    return sp, cfg, worker


def test_play_test_games_is_batch_invariant(monkeypatch):
    """48 games on 48 slots and on 16 slots: the same game ids 0..47 with identical histories; the summary read from
    the packed arrays equals the one of the materialised histories; the next call continues with id 48."""
    monkeypatch.setenv("MZ_TC_MODE", "off")
    out = {}
    for slots in (48, 16):
        sp, cfg, worker = _worker("tictactoe", test_parallel_games=slots)
        games, summary = worker.play_test_games(48, "expert", 1)
        blocks = {int(b["game_id"]): b for b in games.blocks()}
        assert sorted(blocks) == list(range(48)) and summary["num_games"] == 48
        listed = sp.evaluation_summary(list(games), 2, 1)
        assert listed.keys() == summary.keys()
        for k in summary:
            assert summary[k] == listed[k] or (numpy.isnan(summary[k]) and numpy.isnan(listed[k])), k
        out[slots] = (blocks, summary)
        more, _ = worker.play_test_games(4, "expert", 1)
        assert sorted(int(b["game_id"]) for b in more.blocks()) == [48, 49, 50, 51]
        worker.close()
    (a, sa), (b, sb) = out[48], out[16]
    for gid in range(48):
        for key in ("action", "visits", "reward", "to_play", "obs"):
            assert numpy.array_equal(a[gid][key], b[gid][key]), (gid, key)
        assert numpy.array_equal(a[gid]["root_value"], b[gid]["root_value"], equal_nan=True)
    assert sa == sb or all(sa[k] == sb[k] or numpy.isnan(sa[k]) for k in sa)


def test_set_opponent_rejects_bad_arguments():
    from muzero_general_b200.engine import DeviceSelfPlayLoop, debug_opponent_action
    mod, cfg, eng = _engine("tictactoe", 4, 2)
    lib, h = eng.lib, eng._h
    assert lib.mz_selfplay_set_opponent(h, 1, 0) == _lib.MZ_ESTATE                 # no loop yet
    loop = DeviceSelfPlayLoop(eng, "tictactoe", cfg.max_moves)
    assert lib.mz_selfplay_set_opponent(h, 3, 0) == _lib.MZ_EINVAL                 # unknown opponent
    assert lib.mz_selfplay_set_opponent(h, -1, 0) == _lib.MZ_EINVAL
    assert lib.mz_selfplay_set_opponent(h, 1, 2) == _lib.MZ_EINVAL                 # muzero_player not 0 / 1
    assert lib.mz_selfplay_set_opponent(h, 2, -1) == _lib.MZ_EINVAL
    assert lib.mz_selfplay_set_opponent(h, 1, 0) == 0
    assert lib.mz_selfplay_set_opponent(h, 1, 1) == 0                              # plays the opening moves
    assert lib.mz_selfplay_set_opponent(h, 0, 0) == _lib.MZ_ESTATE                 # moves played
    pk = loop.peek()
    assert (pk["move_index"] == 1).all() and (pk["to_play"] == 1).all()
    loop = DeviceSelfPlayLoop(eng, "tictactoe", cfg.max_moves)
    loop.moves(1, 0.0)
    assert lib.mz_selfplay_set_opponent(h, 1, 0) == _lib.MZ_ESTATE                 # moves played
    DeviceSelfPlayLoop(eng, "tictactoe", 1)
    assert lib.mz_selfplay_set_opponent(h, 1, 0) == _lib.MZ_EINVAL                 # max_moves < 2
    DeviceSelfPlayLoop(eng, "tictactoe", cfg.max_moves, td_steps=3, per_alpha=1.0, discount=1.0)
    assert lib.mz_selfplay_set_opponent(h, 2, 0) == _lib.MZ_EINVAL                 # td_steps > 0
    with pytest.raises(ValueError):
        DeviceSelfPlayLoop(eng, "tictactoe", cfg.max_moves, opponent="human")
    eng.close()
    mod, cfg, eng = _engine("cartpole", 4, 2)
    DeviceSelfPlayLoop(eng, "cartpole", 20)
    assert eng.lib.mz_selfplay_set_opponent(eng._h, 1, 0) == _lib.MZ_EINVAL        # one-player game
    assert eng.lib.mz_selfplay_set_opponent(eng._h, 0, 0) == 0
    eng.close()
    board = numpy.zeros((1, 9), numpy.int8)
    with pytest.raises(_lib.MzError):
        debug_opponent_action("tictactoe", "self", board, [1], [0.5])
    assert eng.lib.mz_debug_opponent_action(0, 0, 1, 1, board.ctypes.data, board.ctypes.data, None, None) == _lib.MZ_EINVAL


def test_test_mode_on_the_device_path_leaves_the_self_play_batch_alone(monkeypatch):
    """continuous_self_play(test_mode=True) with test_games_per_report plays on its own engine: the keys are written and
    the worker's training games in flight (its device loop) are exactly where they were."""
    monkeypatch.setenv("MZ_TC_MODE", "off")
    sp, cfg, worker = _worker("tictactoe", training_steps=4, ratio=None, test_games_per_report=20)
    worker.play_moves(3, 1.0)
    before = worker._device_loop.loop.peek()
    steps = worker.env_steps

    class Storage:
        def __init__(self):
            self.d = dict(weights=worker.model.get_weights(), training_step=0, terminate=False)
            self.keys = set()

        def get_info(self, k):
            if k == "training_step":
                self.d["training_step"] += 1
            return self.d[k]

        def set_info(self, k, v=None):
            self.keys |= set(k)
            self.d.update(k)

    storage = Storage()
    worker.continuous_self_play(storage, None, test_mode=True)
    assert storage.keys == {"episode_length", "total_reward", "mean_value", "muzero_reward", "opponent_reward"}
    assert 5 <= storage.d["episode_length"] <= 9 and worker._next_test_game_id >= 20
    after = worker._device_loop.loop.peek()
    assert all(numpy.array_equal(before[k], after[k]) for k in before) and worker.env_steps == steps
    worker.close()
