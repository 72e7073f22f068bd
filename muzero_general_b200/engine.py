"""Python face of the C ABI: one ``SearchEngine`` per GPU process.

``SearchEngine`` owns an ``MzHandle`` and exposes, for a whole batch of games,
what the reference does for one game at a time:

* ``load_weights(state_dict)``          <- ``model.set_weights`` (models.py:72-73)
* ``search(...)``                       <- ``MCTS(config).run`` (self_play.py:260-361)
* ``initial_inference / recurrent_inference``  (models.py:172-195, 601-623)
* ``export_tree(game)``                 <- walking ``Node.children`` (self_play.py:433-449)

All numerical work happens in libmzb200.so; this file only marshals buffers.  Inputs may be
numpy arrays (host memory, copies are part of the call) or CUDA torch tensors (device memory).
"""
from __future__ import annotations

import ctypes as C
import math
from dataclasses import dataclass
from typing import Optional

import numpy

from . import _lib
from .netspec import FC, NetSpec, netspec_from_config, weights_spec


def _is_torch(x):
    return x is not None and type(x).__module__.startswith("torch")


def _fill_layers(desc, prefix, layers):
    if len(layers) > _lib.MZ_MAX_LAYERS:
        raise ValueError(f"at most {_lib.MZ_MAX_LAYERS} hidden layers per head are supported")
    setattr(desc, "n_" + prefix, len(layers))
    arr = getattr(desc, prefix)
    for i, v in enumerate(layers):
        arr[i] = int(v)


def net_desc(spec: NetSpec) -> _lib.MzNetDesc:
    d = _lib.MzNetDesc()
    d.kind = spec.kind
    d.obs_c, d.obs_h, d.obs_w = spec.in_channels, spec.obs_shape[1], spec.obs_shape[2]
    d.action_space = spec.action_space
    d.support_size = spec.support_size
    d.encoding = spec.encoding
    _fill_layers(d, "fc_representation", spec.fc_representation)
    _fill_layers(d, "fc_dynamics", spec.fc_dynamics)
    _fill_layers(d, "fc_reward", spec.fc_reward)
    _fill_layers(d, "fc_value", spec.fc_value)
    _fill_layers(d, "fc_policy", spec.fc_policy)
    d.blocks, d.channels = spec.blocks, spec.channels
    d.reduced_reward, d.reduced_value, d.reduced_policy = spec.reduced_reward, spec.reduced_value, spec.reduced_policy
    _fill_layers(d, "res_fc_reward", spec.res_fc_reward)
    _fill_layers(d, "res_fc_value", spec.res_fc_value)
    _fill_layers(d, "res_fc_policy", spec.res_fc_policy)
    d.downsample = spec.downsample
    return d


@dataclass
class SearchOutput:
    visit_counts: numpy.ndarray          # [n, A] int32
    root_value: numpy.ndarray            # [n] float64
    root_predicted_value: numpy.ndarray  # [n] float32
    max_tree_depth: numpy.ndarray        # [n] int32
    tie_count: numpy.ndarray             # [n] int32
    root_priors: numpy.ndarray           # [n, A] float64
    value_range: numpy.ndarray           # [n, 2] float64
    trace: Optional[dict] = None
    device_ms: float = 0.0


class SearchEngine:
    def __init__(self, config, max_games: int = 1, device: int = 0, seed: Optional[int] = None,
                 num_simulations: Optional[int] = None, extra_expansions: int = 0):
        self.lib = _lib.load_library()
        self.config = config
        self.spec = netspec_from_config(config)
        if list(config.action_space) != list(range(len(config.action_space))):
            raise ValueError("action_space must be list(range(n)) (every reference game file is)")
        if list(config.players) != list(range(len(config.players))):
            raise ValueError("players must be list(range(n))")
        self.A = self.spec.action_space
        self.N = int(config.num_simulations if num_simulations is None else num_simulations)
        self.max_games = int(max_games)
        self.device = int(device)
        self.extra_expansions = int(extra_expansions)       # pool room for searches continued from an imported tree
        self.pool_n = self.N + self.extra_expansions
        s = _lib.MzSearchDesc()
        s.max_games = self.max_games
        s.num_simulations = self.N
        s.extra_expansions = self.extra_expansions
        s.num_players = len(config.players)
        s.discount = float(config.discount)
        s.pb_c_base = float(config.pb_c_base)
        s.pb_c_init = float(config.pb_c_init)
        s.root_dirichlet_alpha = float(config.root_dirichlet_alpha)
        s.root_exploration_fraction = float(config.root_exploration_fraction)
        s.seed = int(config.seed if seed is None else seed) & 0xFFFFFFFFFFFFFFFF
        # math.log / math.sqrt exactly as the reference evaluates them (self_play.py:385-390)
        n = self.pool_n + 2
        self._pbc = (C.c_double * n)(*[math.log((i + config.pb_c_base + 1) / config.pb_c_base) + config.pb_c_init
                                       for i in range(n)])
        self._sqrt = (C.c_double * n)(*[math.sqrt(i) for i in range(n)])
        s.pb_c_table = C.cast(self._pbc, C.POINTER(C.c_double))
        s.sqrt_table = C.cast(self._sqrt, C.POINTER(C.c_double))
        # the whole exploration factor pb_c(n_p) * (sqrt(n_p) / (n_c + 1)) with Python's own roundings
        self._ucb = (C.c_double * (n * n))(*[self._pbc[p] * (self._sqrt[p] / (c + 1)) for p in range(n) for c in range(n)])
        s.ucb_table = C.cast(self._ucb, C.POINTER(C.c_double))
        self._net_desc = net_desc(self.spec)
        handle = C.c_void_p()
        rc = self.lib.mz_create(C.byref(self._net_desc), C.byref(s), self.device, C.byref(handle))
        if rc != 0:
            msg = self.lib.mz_last_error(None).decode()
            if rc == _lib.MZ_EUNSUPPORTED:
                raise NotImplementedError(msg)
            raise _lib.MzError(rc, msg)
        self._h = handle
        self.hidden_elems = int(self.lib.mz_hidden_elems(self._h))
        self.obs_elems = int(self.lib.mz_obs_elems(self._h))

    # ------------------------------------------------------------------ plumbing
    def close(self):
        if getattr(self, "_h", None):
            self.lib.mz_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc):
        if rc != 0:
            raise _lib.MzError(rc, self.lib.mz_last_error(self._h).decode())

    @property
    def launch_count(self):
        return int(self.lib.mz_launch_count(self._h))

    @property
    def graph_partitions(self):
        """Parallel branches of the replayed search graph (1 = one chain of kernels)."""
        return int(self.lib.mz_graph_partitions(self._h))

    @property
    def last_search_ms(self):
        return float(self.lib.mz_last_search_ms(self._h))

    @property
    def numerics(self):
        """Arithmetic of the search path (bench.py's dtype)."""
        return self.lib.mz_numerics(self._h).decode()

    KERNEL_CLASSES = ("tree_step_kernel", "conv_tower_tc_kernel", "heads_kernel", "conv3x3_kernel", "other", "small_tower_kernel",
                      "small_search_kernel")

    def kernel_timing(self, enable):
        """Bracket every kernel of the step-wise pipeline with CUDA events (no graph replay while enabled)."""
        self._check(self.lib.mz_kernel_timing(self._h, 1 if enable else 0))

    def kernel_times(self):
        """{kernel class: (total ms, launches)} since the last call (mz_kernel_times)."""
        import ctypes as C
        ms = (C.c_double * len(self.KERNEL_CLASSES))()
        cnt = (C.c_int64 * len(self.KERNEL_CLASSES))()
        self._check(self.lib.mz_kernel_times(self._h, ms, cnt))
        return {k: (float(ms[i]), int(cnt[i])) for i, k in enumerate(self.KERNEL_CLASSES)}

    @staticmethod
    def _ptr(x, dtype, keep):
        """Pointer of a numpy array (made contiguous, right dtype) or of a CUDA torch tensor."""
        if x is None:
            return None
        if _is_torch(x):
            import torch
            want = {numpy.float32: torch.float32, numpy.float64: torch.float64, numpy.int32: torch.int32,
                    numpy.int64: torch.int64, numpy.uint8: torch.uint8}[dtype]
            if x.dtype != want or not x.is_contiguous():
                x = x.to(want).contiguous()
            keep.append(x)
            return x.data_ptr()
        a = numpy.ascontiguousarray(x, dtype=dtype)
        keep.append(a)
        return a.ctypes.data

    # ------------------------------------------------------------------ weights
    def load_weights(self, state_dict):
        """Accepts the reference ``state_dict`` (torch tensors or numpy arrays, CPU)."""
        tensors, keep = [], []
        for key, shape in weights_spec(self.spec):
            if key.endswith("num_batches_tracked"):
                continue
            if key not in state_dict:
                raise KeyError(f"state_dict is missing {key}")
            v = state_dict[key]
            if _is_torch(v):
                v = v.detach().cpu().numpy()
            a = numpy.ascontiguousarray(v, dtype=numpy.float32)
            if tuple(a.shape) != tuple(shape):
                raise ValueError(f"{key}: expected shape {tuple(shape)}, got {tuple(a.shape)}")
            keep.append(a)
            tensors.append((key.encode(), a))
        arr = (_lib.MzTensor * len(tensors))()
        for i, (name, a) in enumerate(tensors):
            arr[i].name = name
            arr[i].data = a.ctypes.data
            arr[i].numel = a.size
        self._check(self.lib.mz_load_weights(self._h, arr, len(tensors)))

    # ------------------------------------------------------------------ search
    def search(self, obs=None, legal_mask=None, to_play=None, add_exploration_noise=False, noise=None,
               first_index=None, game_id=None, move_index=None, teacher=None, trace=False, trace_depth=None,
               keep_tree=False, stepwise=False, n_games=None, continue_tree=False) -> SearchOutput:
        A, N = self.A, self.N
        keep = []
        if n_games is None:
            src = obs if obs is not None else (teacher["root_value"] if teacher else legal_mask)
            n_games = 1 if (src is None and continue_tree) else int(src.shape[0])
        n = n_games
        device_mem = _is_torch(obs)
        io = _lib.MzSearchIO()
        io.n_games = n
        io.mem = _lib.MZ_MEM_DEVICE if device_mem else _lib.MZ_MEM_HOST
        if obs is not None:
            if not device_mem:
                obs = numpy.asarray(obs, dtype=numpy.float32).reshape(n, -1)
                if obs.shape[1] != self.obs_elems:
                    raise ValueError(f"observation has {obs.shape[1]} elements, expected {self.obs_elems}")
            io.obs = self._ptr(obs, numpy.float32, keep)
        if legal_mask is not None and not _is_torch(legal_mask):
            # the reference asserts this per game (self_play.py:296); a row without a legal action would also
            # index the node pool out of bounds on the device
            assert numpy.asarray(legal_mask).reshape(n, -1).any(axis=1).all(), \
                "Legal actions should not be an empty array."
        io.legal_mask = self._ptr(legal_mask, numpy.uint8, keep)
        io.to_play = self._ptr(to_play, numpy.int32, keep)
        io.add_exploration_noise = int(bool(add_exploration_noise))
        io.flags = ((_lib.MZ_FLAG_KEEP_TREE if keep_tree else 0) | (_lib.MZ_FLAG_STEPWISE if stepwise else 0)
                    | (_lib.MZ_FLAG_CONTINUE if continue_tree else 0))
        io.noise = self._ptr(noise, numpy.float64, keep)
        io.first_index = self._ptr(first_index, numpy.int32, keep)
        io.game_id = self._ptr(game_id, numpy.int64, keep)
        io.move_index = self._ptr(move_index, numpy.int32, keep)

        if device_mem:
            import torch
            dev = obs.device
            mk = lambda shape, dt: torch.empty(shape, dtype=dt, device=dev)
            out = SearchOutput(mk((n, A), torch.int32), mk((n,), torch.float64), mk((n,), torch.float32),
                               mk((n,), torch.int32), mk((n,), torch.int32), mk((n, A), torch.float64),
                               mk((n, 2), torch.float64))
            p = lambda t: t.data_ptr()
        else:
            out = SearchOutput(numpy.empty((n, A), numpy.int32), numpy.empty(n, numpy.float64),
                               numpy.empty(n, numpy.float32), numpy.empty(n, numpy.int32), numpy.empty(n, numpy.int32),
                               numpy.empty((n, A), numpy.float64), numpy.empty((n, 2), numpy.float64))
            p = lambda a: a.ctypes.data
        io.visit_counts, io.root_value, io.root_predicted_value = p(out.visit_counts), p(out.root_value), p(out.root_predicted_value)
        io.max_tree_depth, io.tie_count, io.root_priors = p(out.max_tree_depth), p(out.tie_count), p(out.root_priors)
        io.value_range = p(out.value_range)

        if teacher is not None:
            t = _lib.MzTeacher()
            for f in ("root_value", "root_reward", "root_priors", "value", "reward", "priors"):
                setattr(t, f, self._ptr(teacher[f], numpy.float32, keep))
            keep.append(t)
            io.teacher = C.pointer(t)
        if trace:
            if device_mem:
                raise ValueError("trace is only available with host buffers")
            D = int(trace_depth or max(1, N))
            tr = dict(depth=numpy.zeros((n, N), numpy.int32), actions=numpy.zeros((n, N, D), numpy.uint8),
                      value=numpy.zeros((n, N), numpy.float32), reward=numpy.zeros((n, N), numpy.float32),
                      priors=numpy.zeros((n, N, A), numpy.float32), root_priors_raw=numpy.zeros((n, A), numpy.float32),
                      root_reward=numpy.zeros(n, numpy.float32), noise=numpy.zeros((n, A), numpy.float64))
            t = _lib.MzTrace()
            t.max_depth = D
            for k, v in tr.items():
                setattr(t, k, v.ctypes.data)
            keep.append(t)
            io.trace = C.pointer(t)
            out.trace = tr
        self._check(self.lib.mz_search(self._h, C.byref(io)))
        out.device_ms = self.last_search_ms
        return out

    # ------------------------------------------------------------------ networks
    def _inference(self, fn, n, x, action):
        A, F, H = self.A, self.spec.full_support, self.hidden_elems
        keep = []
        res = dict(value_logits=numpy.empty((n, F), numpy.float32), reward_logits=numpy.empty((n, F), numpy.float32),
                   policy_logits=numpy.empty((n, A), numpy.float32), hidden=numpy.empty((n, H), numpy.float32),
                   value=numpy.empty(n, numpy.float32), reward=numpy.empty(n, numpy.float32))
        o = _lib.MzInferenceOut()
        for k, v in res.items():
            setattr(o, k, v.ctypes.data)
        xp = self._ptr(numpy.asarray(x, dtype=numpy.float32).reshape(n, -1), numpy.float32, keep)
        if action is None:
            self._check(fn(self._h, n, _lib.MZ_MEM_HOST, xp, C.byref(o)))
        else:
            ap = self._ptr(numpy.asarray(action).reshape(n), numpy.int32, keep)
            self._check(fn(self._h, n, _lib.MZ_MEM_HOST, xp, ap, C.byref(o)))
        return res

    def initial_inference(self, obs):
        obs = numpy.asarray(obs, dtype=numpy.float32)
        return self._inference(self.lib.mz_initial_inference, obs.shape[0], obs, None)

    def recurrent_inference(self, hidden, action):
        hidden = numpy.asarray(hidden, dtype=numpy.float32)
        return self._inference(self.lib.mz_recurrent_inference, hidden.shape[0], hidden, action)

    # ------------------------------------------------------------------ tree
    def export_tree(self, game: int, with_hidden: bool = False):
        S = (self.pool_n + 1) * self.A
        out = dict(child_visit=numpy.zeros(S, numpy.int32), child_value_sum=numpy.zeros(S, numpy.float64),
                   child_reward=numpy.zeros(S, numpy.float32), child_prior=numpy.zeros(S, numpy.float64),
                   child_expansion=numpy.full(S, -1, numpy.int32))
        e = _lib.MzTreeExport()
        for k, v in out.items():
            setattr(e, k, v.ctypes.data)
        if with_hidden:
            out["hidden"] = numpy.zeros((self.pool_n + 1, self.hidden_elems), numpy.float32)
            e.hidden = out["hidden"].ctypes.data
        self._check(self.lib.mz_export_tree(self._h, int(game), C.byref(e)))
        out["n_expansions"] = int(e.n_expansions)
        out["root_visit"] = int(e.root_visit)
        out["root_value_sum"] = float(e.root_value_sum)
        out["root_reward"] = float(e.root_reward)
        return out

    def import_tree(self, game: int, tree: dict):
        """Seed game ``game``'s tree in the node pool (the inverse of ``export_tree``; ``mz_import_tree``): arrays
        ``child_visit / child_value_sum / child_reward / child_prior / child_expansion`` of ``n_expansions * A`` entries,
        ``hidden [n_expansions, hidden_elems]``, ``root_visit``, ``root_value_sum``, ``root_reward``."""
        keep = []
        K = int(tree["n_expansions"])
        e = _lib.MzTreeExport()
        e.n_expansions = K
        for k, dt in (("child_visit", numpy.int32), ("child_value_sum", numpy.float64), ("child_reward", numpy.float32),
                      ("child_prior", numpy.float64), ("child_expansion", numpy.int32)):
            a = numpy.ascontiguousarray(tree[k], dtype=dt).reshape(-1)
            assert a.size >= K * self.A, k
            keep.append(a)
            setattr(e, k, a.ctypes.data)
        if tree.get("hidden") is not None:
            hdn = numpy.ascontiguousarray(tree["hidden"], dtype=numpy.float32).reshape(-1)
            assert hdn.size >= K * self.hidden_elems
            keep.append(hdn)
            e.hidden = hdn.ctypes.data
        e.root_visit = int(tree["root_visit"])
        e.root_value_sum = float(tree["root_value_sum"])
        e.root_reward = float(tree.get("root_reward", 0.0))
        self._check(self.lib.mz_import_tree(self._h, int(game), C.byref(e)))


class DeviceSelfPlayLoop:
    """Python face of mz_selfplay_*: ``max_games`` environments stepped on the GPU, one batched search per move,
    finished games handed back as packed struct-of-arrays blocks (SURVEY.md 8f-1, include/mzb200.h)."""

    ENVS = {"cartpole": _lib.MZ_ENV_CARTPOLE, "tictactoe": _lib.MZ_ENV_TICTACTOE, "connect4": _lib.MZ_ENV_CONNECT4}
    OPPONENTS = {"self": _lib.MZ_OPPONENT_SELF, "expert": _lib.MZ_OPPONENT_EXPERT, "random": _lib.MZ_OPPONENT_RANDOM}

    def __init__(self, engine: SearchEngine, env: str, max_moves: int, temperature_threshold=None, reward_scale: int = 1,
                 first_game_id: int = 0, staging_bytes: int = 0, game_id_stride: int = 0, td_steps: int = 0,
                 per_alpha: float = 1.0, discount: float = 1.0, opponent: str = "self", muzero_player: int = 0):
        """``opponent`` = "expert" / "random" plays evaluation games (``mz_selfplay_set_opponent``): MuZero searches the
        moves of side ``muzero_player`` only, the hard-coded opponent plays the other side on the device."""
        if env not in self.ENVS:
            raise NotImplementedError(f"no device-resident environment for {env!r}")
        if opponent not in self.OPPONENTS:
            raise ValueError(f"opponent must be one of {sorted(self.OPPONENTS)}, got {opponent!r}")
        self.engine = engine
        d = _lib.MzSelfPlayDesc()
        d.env = self.ENVS[env]
        d.max_moves = int(max_moves)
        d.temperature_threshold = int(temperature_threshold or 0)
        d.reward_scale = int(reward_scale)
        d.first_game_id = int(first_game_id)
        d.game_id_stride = int(game_id_stride)
        if td_steps and per_alpha in (0.5, 1, 1.0):
            # PER priorities on the device: discount ** k evaluated HERE, with Python's pow, like replay_buffer.py:246,260
            self._discount_pow = (C.c_double * (int(td_steps) + 1))(*[discount ** k for k in range(int(td_steps) + 1)])
            d.td_steps, d.per_alpha = int(td_steps), float(per_alpha)
            d.discount_pow = C.cast(self._discount_pow, C.c_void_p)
        self.with_priorities = bool(d.td_steps)
        d.staging_bytes = int(staging_bytes)
        engine._check(engine.lib.mz_selfplay_begin(engine._h, C.byref(d)))
        if opponent != "self":
            engine._check(engine.lib.mz_selfplay_set_opponent(engine._h, self.OPPONENTS[opponent], int(muzero_player)))
        self.opponent, self.muzero_player = opponent, int(muzero_player)
        self.stats = _lib.MzSelfPlayStats()

    def moves(self, n_moves: int, temperature: float, forced_action=None, uniform=None, noise=None, first_index=None):
        """Play ``n_moves`` lockstep moves; returns the stats struct (env_steps, games_finished, staged_*, device_ms)."""
        eng = self.engine
        inj, keep = None, []
        if forced_action is not None or uniform is not None or noise is not None or first_index is not None:
            inj = _lib.MzSelfPlayInject()
            inj.forced_action = eng._ptr(forced_action, numpy.int32, keep)
            inj.uniform = eng._ptr(uniform, numpy.float64, keep)
            inj.noise = eng._ptr(noise, numpy.float64, keep)
            inj.first_index = eng._ptr(first_index, numpy.int32, keep)
        eng._check(eng.lib.mz_selfplay_moves(eng._h, int(n_moves), float(temperature),
                                            C.byref(inj) if inj is not None else None, C.byref(self.stats)))
        return self.stats

    def enqueue(self, n_moves: int, temperature: float):
        """Start ``n_moves`` moves without waiting (``mz_selfplay_enqueue``); pair with ``wait``."""
        eng = self.engine
        eng._check(eng.lib.mz_selfplay_enqueue(eng._h, int(n_moves), float(temperature)))

    def wait(self):
        eng = self.engine
        eng._check(eng.lib.mz_selfplay_wait(eng._h, C.byref(self.stats)))
        return self.stats

    def drain_pointers(self):
        """(data address, bytes, games, index address) of the staged games, zero-copy.  The library swaps its two staging
        areas here, so the memory stays intact while the next moves run; copy it before the drain after that."""
        eng = self.engine
        ptr, nbytes, ngames, iptr = C.c_void_p(), C.c_uint64(), C.c_int32(), C.c_void_p()
        eng._check(eng.lib.mz_selfplay_drain(eng._h, C.byref(ptr), C.byref(nbytes), C.byref(ngames), C.byref(iptr)))
        return ptr.value, int(nbytes.value), int(ngames.value), iptr.value

    @staticmethod
    def copy_staged(pointers):
        """``drain_pointers()`` -> (bytes, index[n, 2] uint64) copies."""
        ptr, nbytes, n, iptr = pointers
        if n == 0:
            return b"", numpy.zeros((0, 2), numpy.uint64)
        index = numpy.frombuffer(C.string_at(iptr, 16 * n), numpy.uint64).reshape(n, 2)
        return C.string_at(ptr, nbytes), index

    def drain(self):
        """(bytes, index) of the staged finished games - copies.
        ``index`` is an ``[n, 2]`` uint64 array: byte offset of each game's block, ``(slot << 32) | length``."""
        return self.copy_staged(self.drain_pointers())

    def peek(self):
        eng = self.engine
        B, A = eng.max_games, eng.A
        out = dict(obs=numpy.empty((B, eng.obs_elems), numpy.float32), legal_mask=numpy.empty((B, A), numpy.uint8),
                   to_play=numpy.empty(B, numpy.int32), game_id=numpy.empty(B, numpy.int64),
                   move_index=numpy.empty(B, numpy.int32), last_action=numpy.empty(B, numpy.int32))
        pk = _lib.MzSelfPlayPeek()
        for k, v in out.items():
            setattr(pk, k, v.ctypes.data)
        eng._check(eng.lib.mz_selfplay_peek(eng._h, C.byref(pk)))
        return out


def parse_staged_game(buf: bytes, off: int):
    """One packed block of ``mz_selfplay_drain`` -> dict of numpy views into ``buf`` (no copies)."""
    H = _lib.MZ_STAGED_HEADER_BYTES
    gid = int(numpy.frombuffer(buf, numpy.int64, 1, off)[0])
    slot, T, first_to_play, O, A, nbytes = (int(x) for x in numpy.frombuffer(buf, numpy.int32, 6, off + 8))
    p = off + H
    root = numpy.frombuffer(buf, numpy.float64, T, p); p += 8 * T
    visits = numpy.frombuffer(buf, numpy.int32, T * A, p).reshape(T, A); p += 4 * T * A
    action = numpy.frombuffer(buf, numpy.int32, T, p); p += 4 * T
    reward = numpy.frombuffer(buf, numpy.float32, T, p); p += 4 * T
    to_play = numpy.frombuffer(buf, numpy.int32, T, p); p += 4 * T
    priority = numpy.frombuffer(buf, numpy.float32, T, p); p += 4 * T
    obs = numpy.frombuffer(buf, numpy.float32, (T + 1) * O, p).reshape(T + 1, O)
    return dict(game_id=gid, slot=slot, length=T, first_to_play=first_to_play, root_value=root, visits=visits,
                action=action, reward=reward, to_play=to_play, priority=priority, obs=obs, bytes=nbytes)


def parse_staged_games(buf: bytes, index):
    """All staged games of one drain, in staging order."""
    games = [parse_staged_game(buf, int(off)) for off in index[:, 0]]
    assert sum(g["bytes"] for g in games) == len(buf), "staged blocks do not add up"
    for g, meta in zip(games, index[:, 1]):
        assert (int(meta) >> 32, int(meta) & 0xFFFFFFFF) == (g["slot"], g["length"])
    return games


def debug_opponent_action(env, opponent, board, player, uniform, device=0):
    """The device's hard-coded opponent (``mz_debug_opponent_action``, the function the evaluation loop plays with) on n
    positions: ``env`` "tictactoe" / "connect4", ``opponent`` "expert" / "random", ``board`` [n, H*W] (+1 / -1 / 0, row 0
    at the bottom), ``player`` [n] side to move (+1 / -1), ``uniform`` [n] the default move's draw.  Returns int32 [n]."""
    lib = _lib.load_library()
    board = numpy.ascontiguousarray(board, numpy.int8)
    n = board.shape[0]
    player = numpy.ascontiguousarray(player, numpy.int8).reshape(n)
    uniform = numpy.ascontiguousarray(uniform, numpy.float64).reshape(n)
    out = numpy.empty(n, numpy.int32)
    rc = lib.mz_debug_opponent_action(device, DeviceSelfPlayLoop.ENVS[env], DeviceSelfPlayLoop.OPPONENTS[opponent], n,
                                      board.ctypes.data, player.ctypes.data, uniform.ctypes.data, out.ctypes.data)
    if rc != 0:
        raise _lib.MzError(rc, lib.mz_last_error(None).decode())
    return out


def debug_conv3x3(x, w, bias=None, residual=None, relu=False, tensor_cores=False, device=0):
    """One conv3x3 (pad 1, stride 1) on the device through mz_debug_conv3x3; numpy NCHW in and out.
    ``tensor_cores``: False / "off" = CUDA cores, "fp16" = tcgen05 with fp16 operands, True / "x3" = tcgen05 split operands."""
    lib = _lib.load_library()
    x = numpy.ascontiguousarray(x, numpy.float32)
    w = numpy.ascontiguousarray(w, numpy.float32)
    n, Cc, H, W = x.shape
    out = numpy.empty_like(x)
    b = None if bias is None else numpy.ascontiguousarray(bias, numpy.float32)
    r = None if residual is None else numpy.ascontiguousarray(residual, numpy.float32)
    mode = {False: 0, True: 2, "off": 0, "fp16": 1, "x3": 2}[tensor_cores]
    rc = lib.mz_debug_conv3x3(device, n, Cc, H, W, x.ctypes.data, w.ctypes.data, None if b is None else b.ctypes.data,
                              None if r is None else r.ctypes.data, int(relu), mode, out.ctypes.data)
    if rc != 0:
        raise _lib.MzError(rc, lib.mz_last_error(None).decode())
    return out
