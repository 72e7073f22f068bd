"""Bulk callers either side of the self-play path (muzero_general_b200/reanalyse.py) on the CPU: PER priorities against
those the unmodified reference ReplayBuffer computed (recorded golden data), batched Reanalyse against the oracle network."""
import copy

import numpy
import pytest
import torch

from conftest import golden_json, weights_for
from fake_engine import FakeSearchEngine
from helpers import random_history
from muzero_general_b200 import reanalyse as ra
from muzero_general_b200.games import load_game_module
from muzero_general_b200.netspec import netspec_from_config
from oracle.gen_golden import PRIORITY_CASES, PRIORITY_LENGTHS, priority_key

torch.set_num_threads(1)


class _RecordingBuffer:
    def __init__(self):
        self.saved = []

    def save_game(self, game_history, shared_storage=None):
        self.saved.append(game_history)


@pytest.mark.parametrize("name,td,discount,alpha,reanalysed", PRIORITY_CASES)
def test_bulk_priorities_equal_the_reference_save_game(name, td, discount, alpha, reanalysed):
    """initial_priorities == what the unmodified ReplayBuffer.save_game computes, bit for bit (float32 priorities, game
    priority; recorded in tests/golden/replay_buffer.json by oracle/gen_golden.py --replay), for one- and two-player
    games, with and without reanalysed values, short and long td horizons."""
    want = golden_json("replay_buffer.json")["priorities"][priority_key(name, td, discount, alpha, reanalysed)]
    cfg = load_game_module(name).MuZeroConfig()
    cfg.td_steps, cfg.discount, cfg.PER_alpha, cfg.PER = td, discount, alpha, True
    rs = numpy.random.RandomState(4)
    assert [w["T"] for w in want] == list(PRIORITY_LENGTHS)
    for T, w in zip(PRIORITY_LENGTHS, want):
        gh = random_history(rs, cfg, T, len(cfg.players))
        if reanalysed:
            gh.reanalysed_predicted_root_values = rs.standard_normal(T).astype(numpy.float32)
        theirs = numpy.array(w["priorities"], dtype=numpy.float32)
        assert numpy.array_equal(theirs, w["priorities"])               # the fixture holds float32 values exactly
        mine, top = ra.initial_priorities(copy.deepcopy(gh), cfg)
        assert mine.dtype == numpy.float32
        assert numpy.array_equal(mine, theirs), (name, T)
        assert top == w["game_priority"]
        # and save_games attaches them before the buffer's save_game sees the game (which then keeps them as they are)
        buf = _RecordingBuffer()
        ra.save_games(buf, [copy.deepcopy(gh)], cfg)
        assert len(buf.saved) == 1 and numpy.array_equal(buf.saved[0].priorities, theirs)
        assert buf.saved[0].game_priority == w["game_priority"]


def test_batched_reanalyse_matches_per_game_inference(monkeypatch):
    """One batched call over many games == the reference's per-game computation (replay_buffer.py:345-366) done with
    the oracle network; the actor loop updates the buffer and the counter."""
    from oracle.net import OracleNet, support_to_scalar
    monkeypatch.setattr(ra, "SearchEngine", FakeSearchEngine)
    mod = load_game_module("tictactoe")
    cfg = mod.MuZeroConfig()
    cfg.training_steps = 3
    spec = netspec_from_config(cfg)
    w = weights_for("tictactoe", spec)
    rs = numpy.random.RandomState(2)
    games = [random_history(rs, cfg, T, 2) for T in (1, 5, 9, 3)]
    for g in games:
        g.observation_history = [rs.randint(0, 2, cfg.observation_shape).astype(numpy.int32) for _ in g.observation_history]
    actor = ra.Reanalyse({"weights": w, "num_reanalysed_games": 0}, cfg, max_positions=7)      # forces several chunks
    actor.reanalyse_games(games)
    net = OracleNet(spec, w)
    for g in games:
        T = len(g.root_values)
        obs = numpy.array([g.get_stacked_observations(i, cfg.stacked_observations, 9) for i in range(T)], dtype=numpy.float32)
        want = torch.squeeze(support_to_scalar(net.initial_inference(obs)[0], cfg.support_size)).numpy()
        assert g.reanalysed_predicted_root_values.shape == want.shape and g.reanalysed_predicted_root_values.dtype == numpy.float32
        numpy.testing.assert_allclose(g.reanalysed_predicted_root_values, want, rtol=1e-6, atol=1e-7)
    assert actor.num_reanalysed_games == 4

    class Storage:
        def __init__(self):
            self.d = dict(weights=w, training_step=0, terminate=False, num_played_games=4, num_reanalysed_games=0)
        def get_info(self, k):
            if k == "training_step":
                self.d[k] += 1
            return self.d[k]
        def set_info(self, k, v=None):
            self.d.update(k if isinstance(k, dict) else {k: v})

    class Buffer:
        def __init__(self):
            self.buffer = {i: copy.deepcopy(g) for i, g in enumerate(games)}
            self.updated = set()
        def sample_game(self, force_uniform=False):
            i = int(rs.randint(len(self.buffer)))
            return i, self.buffer[i], None
        def update_game_history(self, game_id, gh):
            self.updated.add(game_id); self.buffer[game_id] = gh

    st, buf = Storage(), Buffer()
    actor.games_per_call = 3
    actor.reanalyse(buf, st)
    assert buf.updated and st.d["num_reanalysed_games"] == actor.num_reanalysed_games > 4
