"""Lookahead selection of the fused FC search kernel (tree.cuh::tree_select_lookahead).

With |A| <= 2 the kernel scores K tree levels per selection round (K = 2, 3, 4 at lane groups of 8, 16, 32) and resolves
the path from one ballot.  MZ_FC_LOOKAHEAD=0 forces the one-level-per-round loop.  Both must give the same search, bit for
bit: the same visit counts, root values, value ranges, tie counts, selected paths and trees."""
import numpy
import pytest

from conftest import weights_for
from muzero_general_b200.netspec import netspec_from_config

pytestmark = pytest.mark.gpu


def _engine(cfg, n, N):
    from muzero_general_b200.engine import SearchEngine
    return SearchEngine(cfg, max_games=n, num_simulations=N)


@pytest.mark.parametrize("wname", ["cartpole", "cartpole_pretrained"])
def test_lookahead_matches_per_level_selection(wname, game_configs, monkeypatch):
    """Headline shape (4096 games, N = 50, device-drawn Dirichlet noise), own networks: lookahead on and off agree."""
    cfg = game_configs["cartpole"]
    spec = netspec_from_config(cfg)
    n, N = 4096, 50
    rs = numpy.random.RandomState(5)
    obs = rs.uniform(-0.05, 0.05, size=(n, 4)).astype(numpy.float32)
    eng = _engine(cfg, n, N)
    eng.load_weights(weights_for(wname, spec))
    outs, trees = [], []
    for la in ("0", "1"):
        monkeypatch.setenv("MZ_FC_LOOKAHEAD", la)
        outs.append(eng.search(obs=obs, add_exploration_noise=True, trace=True, keep_tree=True))
        trees.append([eng.export_tree(i, with_hidden=True) for i in (0, 1, 777, n // 2, n - 1)])
    eng.close()
    a, b = outs
    for f in ("visit_counts", "root_value", "root_predicted_value", "max_tree_depth", "tie_count", "root_priors",
              "value_range"):
        assert numpy.array_equal(getattr(a, f), getattr(b, f)), f
    for f in ("depth", "actions", "value", "reward", "priors"):
        assert numpy.array_equal(a.trace[f], b.trace[f]), f
    assert a.max_tree_depth.max() > 3          # paths do cross round boundaries
    for ta, tb in zip(*trees):
        for k in ta:
            assert numpy.array_equal(numpy.asarray(ta[k]), numpy.asarray(tb[k])), k


@pytest.mark.parametrize("group", ["8", "16", "32"])
def test_lookahead_teacher_forced_ties_vs_c_oracle(group, game_configs, monkeypatch):
    """Teacher-forced |A| = 2 with equal priors and quantised values: exact ties at every depth, so every level position
    of a round resolves ties (Philox draws keyed by the true depth).  Random legal root masks.  Every game equals the C
    oracle bit for bit; the per-level loop gives the same."""
    from oracle import build_c
    monkeypatch.setenv("MZ_FC_GROUP", group)
    cfg = game_configs["cartpole"]
    A, P, n, N, D = 2, 1, 2048, 50, 50
    rs = numpy.random.RandomState(int(group))
    legal = numpy.ones((n, A), numpy.uint8)
    one = rs.uniform(size=n) < 0.3
    legal[one, rs.randint(0, A, n)[one]] = 0                  # 30 % of the roots have a single legal action
    t = dict(root_value=(rs.randint(-2, 3, n) / 4).astype(numpy.float32),
             root_reward=numpy.zeros(n, numpy.float32),
             value=(rs.randint(-2, 3, (n, N)) / 4).astype(numpy.float32),
             reward=(rs.randint(0, 2, (n, N)) / 2).astype(numpy.float32),
             priors=numpy.full((n, N, A), 0.5, numpy.float32))
    t["root_priors"] = (legal / legal.sum(1, keepdims=True)).astype(numpy.float32)
    noise = legal / legal.sum(1, keepdims=True)               # mixing equal noise into equal priors keeps them equal
    to_play = numpy.zeros(n, numpy.int32)
    gid = rs.randint(0, 1 << 40, n).astype(numpy.int64)
    mv = rs.randint(0, 400, n).astype(numpy.int32)
    first = rs.randint(-1, A, n).astype(numpy.int32)
    ref = build_c.tree_search(n, N, A, P, cfg.discount, cfg.pb_c_base, cfg.pb_c_init, cfg.root_exploration_fraction,
                              legal, to_play, noise, first, cfg.seed, gid, mv, t, D=D)
    assert ref["ties"].sum() > 10 * n and ref["max_depth"].max() >= 8
    eng = _engine(cfg, n, N)
    outs = []
    for la in ("1", "0"):
        monkeypatch.setenv("MZ_FC_LOOKAHEAD", la)
        outs.append(eng.search(legal_mask=legal, to_play=to_play, add_exploration_noise=True, noise=noise,
                               first_index=first, game_id=gid, move_index=mv, teacher=t, trace=True, trace_depth=D,
                               n_games=n))
    eng.close()
    mask = numpy.arange(D)[None, None, :] < ref["depth"][:, :, None]
    for out in outs:
        assert (out.visit_counts == ref["visit_counts"]).all()
        assert (out.root_value == ref["root_value"]).all()
        assert (out.max_tree_depth == ref["max_depth"]).all()
        assert (out.tie_count == ref["ties"]).all()
        assert (out.value_range == ref["range"]).all()
        assert (out.trace["depth"] == ref["depth"]).all()
        assert (numpy.where(mask, out.trace["actions"], 0) == numpy.where(mask, ref["actions"], 0)).all()
