#!/usr/bin/env python
"""bench.py - self-play throughput (BASELINE.json metric: env-steps/s and MCTS simulations/s) on N B200s.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--workload NAME] [--impl ours|reference]
                  [--extras a,b,c | --no-extras] [--no-cpu-baseline] [--no-loop] [--dump-outputs DIR]

What is timed
-------------
One SEARCH = the hot path over one batch: a batched MCTS.run (root inference + num_simulations x {select, recurrent
inference, expand, backup}) for every game of the batch = one env-step's worth of search per game.  One STEP =
`searches_per_step` searches over different synthetic batches, chosen so that K steps last >= 1 s (a 0.6 ms CartPole
search would otherwise give a 12 ms sample); the L2 is flushed (256 MiB write, untimed) before every search.
`value` = env-steps/s of search with the inputs resident in HBM (search only - the environment step is NOT in it);
`e2e`   = the same through the C ABI with pinned HOST buffers, H2D + D2H inside the timed region;
`loop`  = env-steps/s of the WHOLE self-play loop through the public `SelfPlay` API (SURVEY.md 8d's full definition:
          search + environment step + action sampling + GameHistory hand-over), timed >= 1 s;
`workloads` = the same sub-lines for the other BASELINE configs at this --gpus N.

--dump-outputs DIR writes what the last timed search of the headline workload returned (visit counts, root values,
root priors, ...; the search's SearchOutput arrays) as DIR/<name>.npy.  Inputs, weights and the search seed are fixed,
and the last timed search always runs on the same one of the rotating input batches, so two runs with the same
arguments, or two builds of the project, can be compared output for output.

N=1 headline workload: BASELINE.json configs[1] - CartPole, fully-connected net, num_simulations=50, 4096 parallel
games per GPU (weak scaling: every rank owns its own games; no data-path collective - one all-gather of per-rank
counters per reporting step, `muzero_general_b200.parallel.gather_counters`).
"""
import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

import numpy

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (game, games per GPU, num_simulations, algorithmic tree+hidden bytes per simulation (SURVEY.md 8d))
    "cartpole_b4096_n50": ("cartpole", 4096, 50, 633.0),
    "cartpole_b4096_n25": ("cartpole", 4096, 25, 530.0),
    "tictactoe_b8192_n50": ("tictactoe", 8192, 50, 2420.0),
    "connect4_b1024_n200": ("connect4", 1024, 200, 22300.0),
    "breakout_b128_n50": ("breakout", 128, 50, 5100.0),
}
DEFAULT_WORKLOAD = "cartpole_b4096_n50"
DEFAULT_EXTRAS = ["connect4_b1024_n200", "connect4_b1024_n200@fp16", "connect4_b1024_n200@off", "tictactoe_b8192_n50", "breakout_b128_n50"]
MIN_TIMED_SECONDS = 1.0

# algorithmic FLOPs of initial_inference / recurrent_inference per sample (SURVEY.md section 8 table)
NET_FLOPS = {"cartpole": (1312.0, 2752.0), "tictactoe": (1.880e5, 2.315e5), "connect4": (3.737e7, 4.040e7),
             "breakout": (3.419e7, 1.532e6)}


def load_peaks():
    """(HBM GB/s, dense bf16 TFLOP/s, which) from the driver-written MEASURED_PEAKS.json, else the fallback."""
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), float(d.get("bf16_tflops_sustained", d["bf16_tflops"])), "measured"
    return 6650.0, 1400.0, "fallback"


def load_traffic():
    """Measured DRAM bytes per launch of the dominant kernels, from the committed ncu captures (profiles/traffic.json)."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    try:
        return json.load(open(p))
    except (OSError, ValueError):
        return {}


def conv3x3_flops(spec, N):
    """FLOPs of the 3x3 convolutions of one search per game: initial_inference + N recurrent_inferences (models.py)."""
    C, blocks = spec.channels, spec.blocks
    obs_c, (_, H, W) = spec.in_channels, spec.obs_shape
    total = 0.0
    if spec.downsample:
        conv = lambda h, w, ci, co: 2.0 * h * w * ci * co * 9
        h1, w1 = (H + 1) // 2, (W + 1) // 2
        total += conv(h1, w1, obs_c, C // 2) + 2 * 2 * conv(h1, w1, C // 2, C // 2)
        h2, w2 = (h1 + 1) // 2, (w1 + 1) // 2
        total += conv(h2, w2, C // 2, C) + 3 * 2 * conv(h2, w2, C, C)
        h3, w3 = (h2 + 1) // 2, (w2 + 1) // 2
        total += 3 * 2 * conv(h3, w3, C, C)
        H, W = (h3 + 1) // 2, (w3 + 1) // 2
    else:
        total += 2.0 * H * W * obs_c * C * 9
    block = 2 * 2.0 * H * W * C * C * 9
    total += 2 * blocks * block                                        # representation + prediction towers
    total += N * (2.0 * H * W * (C + 1) * C * 9 + 2 * blocks * block)  # dynamics stem + dynamics / prediction towers
    return total


# ----------------------------------------------------------------------------- clocks
class ClockSampler:
    QUERY = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.samples = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.QUERY}", "--format=csv,noheader,nounits",
                 "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.samples.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for s in self.samples:
            f = [x.strip() for x in s.split(",")]
            if len(f) < 6:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for nme, v in zip(names, f[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(nme)
        return {"sm_mhz": float(numpy.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ----------------------------------------------------------------------------- CPU arm (oracle port)
def physical_cores():
    """One logical CPU per physical core inside this process's affinity set (SMT siblings dropped)."""
    try:
        allowed = sorted(os.sched_getaffinity(0))
    except AttributeError:
        return list(range(os.cpu_count() or 1))
    seen, out = set(), []
    for c in allowed:
        try:
            sib = open(f"/sys/devices/system/cpu/cpu{c}/topology/thread_siblings_list").read().strip()
        except OSError:
            sib = str(c)
        if sib not in seen:
            seen.add(sib)
            out.append(c)
    return out or allowed


_CPU = {}


def _cpu_init(game, n_sim, cpus, counter):
    """Pool initializer: pin this worker to its own physical core, build the oracle network once."""
    import torch
    torch.set_num_threads(1)
    with counter.get_lock():
        idx = counter.value
        counter.value += 1
    try:
        os.sched_setaffinity(0, {cpus[idx % len(cpus)]})
    except (AttributeError, OSError):
        pass
    from muzero_general_b200.games import load_game_module
    from muzero_general_b200.netspec import netspec_from_config, synthetic_weights
    from oracle import mcts as om
    from oracle.net import OracleNet
    cfg = load_game_module(game).MuZeroConfig()
    spec = netspec_from_config(cfg)
    net = OracleNet(spec, synthetic_weights(spec, 0))
    rs = numpy.random.RandomState(1000 + idx)
    _CPU.update(game=game, spec=spec, rs=rs, draws=om.LegacyNumpyDraws(rs),
                search=om.TreeSearch(om.SearchParams.from_config(cfg, n_sim)),
                ev=om.ModelEvaluator(net, spec.support_size),
                shape=(spec.in_channels,) + tuple(spec.obs_shape[1:]), legal=list(range(spec.action_space)))
    _cpu_one()                 # warm-up


def _cpu_one():
    c = _CPU
    if c["game"] == "cartpole":
        obs = c["rs"].uniform(-0.05, 0.05, size=c["shape"]).astype(numpy.float32)
    else:
        obs = c["rs"].random_sample(c["shape"]).astype(numpy.float32)
    c["search"].run(c["ev"], obs, c["legal"], 0, True, c["draws"])


def _cpu_run(seconds):
    t0 = time.perf_counter()
    done = 0
    while time.perf_counter() - t0 < seconds:
        _cpu_one()
        done += 1
    return done, time.perf_counter() - t0


class CpuArm:
    """The oracle port of the reference's batch-1 Python/torch MCTS.run, one pinned process per physical core.
    The pool is created once (importing torch in 64+ fresh processes costs more than the measurement)."""

    def __init__(self, game, n_sim):
        import multiprocessing as mp
        self.cpus = physical_cores()
        ctx = mp.get_context("spawn")
        self.pool = ctx.Pool(len(self.cpus), initializer=_cpu_init, initargs=(game, n_sim, self.cpus, ctx.Value("i", 0)))

    @property
    def cores(self):
        return len(self.cpus)

    def run(self, seconds):
        res = self.pool.map(_cpu_run, [seconds] * len(self.cpus), chunksize=1)
        searches = sum(r[0] for r in res)
        wall = max(r[1] for r in res)
        return searches / wall, searches, wall

    def close(self):
        self.pool.close()
        self.pool.join()


# ----------------------------------------------------------------------------- distributed helpers
class Dist:
    def __init__(self, dist, dev):
        self.dist, self.dev = dist, dev

    def barrier(self):
        import torch
        if self.dist is not None:
            self.dist.barrier()
        torch.cuda.synchronize()

    def max(self, values):
        import torch
        t = torch.tensor(list(values), dtype=torch.float64, device=self.dev)
        if self.dist is not None:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return [float(x) for x in t.tolist()]


def percentiles(ms):
    a = numpy.asarray(ms, dtype=numpy.float64)
    return {"median": float(numpy.median(a)), "p10": float(numpy.percentile(a, 10)), "p90": float(numpy.percentile(a, 90)),
            "min": float(a.min()), "max": float(a.max()), "count": int(a.size)}


# ----------------------------------------------------------------------------- one workload on this rank
def run_workload(name, args, D, rank, local_rank, world, with_loop, headline):
    """Times one workload on this rank (collectively with the other ranks); returns the sub-line on every rank."""
    import torch
    from muzero_general_b200.engine import SearchEngine
    from muzero_general_b200.games import load_game_module
    from muzero_general_b200.netspec import netspec_from_config, synthetic_weights
    from muzero_general_b200 import parallel

    base, _, mode = name.partition("@")
    game, B, N, bytes_per_sim = WORKLOADS[base]
    prev_mode = os.environ.get("MZ_TC_MODE")
    if mode:
        os.environ["MZ_TC_MODE"] = mode
    dev = torch.device("cuda", local_rank)
    cfg = load_game_module(game).MuZeroConfig()
    spec = netspec_from_config(cfg)
    A = spec.action_space
    eng = SearchEngine(cfg, max_games=B, device=local_rank, num_simulations=N, seed=cfg.seed + rank)
    eng.load_weights(synthetic_weights(spec, 0))
    numerics = eng.numerics if hasattr(eng, "numerics") else "f32"

    # synthetic inputs, a different batch every search (global game ids keep streams rank-independent)
    n_batches = 4
    rs = numpy.random.RandomState(100 + rank)
    shape = (B, eng.obs_elems)
    if game == "cartpole":
        host_obs = [rs.uniform(-0.05, 0.05, size=shape).astype(numpy.float32) for _ in range(n_batches)]
    else:
        host_obs = [rs.random_sample(shape).astype(numpy.float32) for _ in range(n_batches)]
    host_noise = [rs.dirichlet([cfg.root_dirichlet_alpha] * A, size=B) for _ in range(n_batches)]
    pin = lambda a: torch.from_numpy(a).pin_memory()
    pinned_obs = [pin(a) for a in host_obs]
    pinned_noise = [pin(a) for a in host_noise]
    dev_obs = [t.to(dev) for t in pinned_obs]
    dev_noise = [t.to(dev) for t in pinned_noise]
    game_id = (rank * B + numpy.arange(B)).astype(numpy.int64)
    dev_gid = torch.from_numpy(game_id).to(dev)
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)

    def search_device(i):
        return eng.search(obs=dev_obs[i % n_batches], add_exploration_noise=True, noise=dev_noise[i % n_batches],
                          game_id=dev_gid)

    def search_host(i):
        return eng.search(obs=pinned_obs[i % n_batches].numpy(), add_exploration_noise=True,
                          noise=pinned_noise[i % n_batches].numpy(), game_id=game_id)

    def one(fn, i):
        flush.fill_(i & 0xFF)                      # evict L2 before every timed search (untimed)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        out = fn(i)                                # mz_search synchronises its stream before returning
        torch.cuda.synchronize()
        return time.perf_counter() - t0, out

    def timed(fn, steps, warmup):
        est = 0.0
        for i in range(warmup):
            est, _ = one(fn, i)
        # every rank times the same number of searches: K steps x `inner` searches, >= MIN_TIMED_SECONDS in total
        est = D.max([est])[0]
        inner = max(1, int(math.ceil(MIN_TIMED_SECONDS / max(est * steps, 1e-9))))
        D.barrier()
        per_search, per_step, kern, out = [], [], 0.0, None
        i = -(steps * inner) % n_batches          # the last timed search runs on the last batch, whatever `inner` is
        for _ in range(steps):
            acc = 0.0
            for _ in range(inner):
                dt, out = one(fn, i)
                i += 1
                acc += dt
                per_search.append(1000.0 * dt)
                kern += out.device_ms
            per_step.append(1000.0 * acc)
        D.barrier()
        return dict(wall=sum(per_step) / 1000.0, kern_ms=kern, searches=steps * inner, inner=inner,
                    per_search=per_search, per_step=per_step, last=out)

    clocks = ClockSampler(local_rank) if headline else None
    if clocks:
        clocks.start()
    launches0 = eng.launch_count
    # the library replays a search from a CUDA graph once it has seen an argument set twice; the device arm rotates
    # n_batches input buffers, so its warm-up covers every buffer three times (eager, eager, capture) - untimed, like W
    dv = timed(search_device, args.steps, max(args.warmup, 3 * n_batches))
    launches = eng.launch_count - launches0
    graph_parts = eng.graph_partitions
    clk = clocks.stop() if clocks else None
    if headline and rank == 0 and args.dump_outputs:
        dump_outputs(dv["last"], args.dump_outputs)
    hv = timed(search_host, args.steps, args.warmup)
    assert int(numpy.asarray(hv["last"].visit_counts).sum()) == B * N
    kernel_split = {}
    if game != "cartpole":
        eng.kernel_timing(True)
        eng.kernel_times()
        flush.fill_(7)
        torch.cuda.synchronize()
        search_device(0)
        kernel_split = eng.kernel_times()
        eng.kernel_timing(False)

    # slowest rank's time; ONE all-gather of the per-rank counters of this reporting step
    wall, wall_e2e, kern_ms = D.max([dv["wall"], hv["wall"], dv["kern_ms"]])
    table, totals = parallel.gather_counters(D.dist, 0, B * dv["searches"], B * dv["searches"] * N, device=dev)
    total_steps = totals[1]
    hbm_peak, bf16_peak, peak_kind = load_peaks()
    traffic = load_traffic()
    value = total_steps / wall
    kern_s = kern_ms / 1000.0 / dv["searches"]
    if game == "cartpole":
        # dominant kernel: the fused search kernel, one launch per search (SURVEY 8d: HBM roofline)
        alg_bytes = B * (N * bytes_per_sim + eng.obs_elems * 4 + A * 8 + A * 4 + 8)
        achieved = alg_bytes / kern_s / 1e9
        tr = traffic.get("fc_search_kernel", {})
        roofline = {"bound": "hbm", "achieved": achieved, "peak": hbm_peak, "unit": "GB/s",
                    "frac": achieved / hbm_peak, "traffic": tr.get("dram_bytes_per_launch"), "traffic_source": tr.get("source"),
                    "peak_kind": peak_kind, "kernel": "fc_search_kernel", "algorithmic_bytes_per_launch": alg_bytes,
                    "avg_launch_us": 1e6 * kern_s,
                    "note": "tree + hidden states live in shared memory for FC nets: measured DRAM traffic is a fraction "
                            "of the algorithmic bytes, the kernel is issue/latency-bound, not HBM-bound"}
    else:
        # residual nets: tensor roofline (SURVEY 8d) for the dominant kernel, timed live with CUDA event pairs around every
        # launch of one extra (untimed) search (mz_kernel_timing); algorithmic FLOPs = the 3x3 convolutions that kernel class
        # executes in one search (2*H*W*Cin*Cout*9 each).  Tensor peak = the measured dense bf16 figure whatever the operand
        # split (the x3 mode issues 3 MMAs per algorithmic MMA: its useful-FLOP fraction is reported, not its issue rate).
        f0, f1 = NET_FLOPS[game]
        flops = B * (f0 + N * f1)
        conv_flops = B * conv3x3_flops(spec, N)
        split = {k: {"ms": v[0], "launches": v[1]} for k, v in kernel_split.items() if v[1]}
        total_ms = sum(v["ms"] for v in split.values()) or 1.0
        for v in split.values():
            v["share"] = v["ms"] / total_ms
        conv_classes = [k for k in ("conv_tower_tc_kernel", "small_search_kernel", "small_tower_kernel", "conv3x3_kernel") if k in split]
        dominant = max(conv_classes, key=lambda k: split[k]["ms"]) if conv_classes else "other"
        conv_ms = sum(split[k]["ms"] for k in conv_classes) or total_ms
        dom = split.get(dominant, {"ms": total_ms, "launches": 1})
        # the dominant class's share of the conv FLOPs ~ its share of the conv time is NOT assumed: classes other than the
        # dominant one only run the stem / DownSample convs, a few % of the FLOPs; achieved uses ALL conv FLOPs over ALL conv time
        achieved = conv_flops / (conv_ms / 1000.0) / 1e12
        tr = traffic.get(f"{dominant}:{game}@{mode}" if mode else f"{dominant}:{game}") or \
            traffic.get(f"{dominant}:{game}" if not mode else "", {}) or {}
        roofline = {"bound": "tensor", "achieved": achieved, "peak": bf16_peak, "unit": "TFLOP/s",
                    "frac": achieved / bf16_peak, "traffic": tr.get("dram_bytes_per_launch"), "traffic_source": tr.get("source"),
                    "peak_kind": peak_kind + " dense bf16 (sustained)",
                    "kernel": dominant, "launches_per_search": dom["launches"],
                    "avg_launch_us": 1000.0 * dom["ms"] / max(dom["launches"], 1),
                    "algorithmic_flops_per_launch": conv_flops / max(dom["launches"], 1),
                    "kernel_split": split,
                    "step_level": {"algorithmic_flops_per_search": flops, "achieved": flops / kern_s / 1e12,
                                   "frac": flops / kern_s / 1e12 / bf16_peak}}
    sub = {
        "workload": name, "value": value, "unit": "env-steps/s", "sims_per_sec": value * N,
        "value_is": "search only (no environment step); see loop",
        "dtype": numerics, "games_per_gpu": B, "num_simulations": N,
        "graph_branches": graph_parts,        # parallel branches of the replayed search graph (partitioned replay); 1 = one chain
        "steps": args.steps, "searches_per_step": dv["inner"], "ms_per_step": 1000.0 * wall / args.steps,
        "ms_per_search": percentiles(dv["per_search"]), "timed_seconds": wall,
        "kernel_ms_per_search": kern_ms / dv["searches"],
        "e2e": {"value": B * world * hv["searches"] / wall_e2e, "unit": "env-steps/s",
                "h2d_bytes_per_step": int(hv["inner"] * B * (eng.obs_elems * 4 + A * 8 + 8)),
                "d2h_bytes_per_step": int(hv["inner"] * B * (A * 4 + 8 + 4 + 4 + 4 + A * 8 + 16)),
                "ms_per_search": percentiles(hv["per_search"]), "searches_per_step": hv["inner"]},
        "gpu_launches": int(launches), "roofline": roofline, "per_rank_counters": table,
    }
    if clk:
        sub["clocks"] = clk
    eng.close()
    if headline and game == "cartpole" and world == 1 and not args.no_saturation:
        sub["saturation"] = saturation_curve(cfg, spec, N, local_rank, dev)
    del flush, dev_obs, dev_noise
    torch.cuda.empty_cache()
    if with_loop:
        try:
            sub["loop"] = selfplay_loop(game, B, N, local_rank, rank, world, D)
        except Exception as e:                           # never lose the line over the loop measurement
            sub["loop"] = {"error": repr(e)}
    if mode:
        if prev_mode is None:
            os.environ.pop("MZ_TC_MODE", None)
        else:
            os.environ["MZ_TC_MODE"] = prev_mode
    return sub


DUMP_FIELDS = ("visit_counts", "root_value", "root_predicted_value", "max_tree_depth", "tie_count", "root_priors",
               "value_range")
DUMP_MAX_BYTES = 64 << 20


def dump_outputs(out, directory):
    """Writes the SearchOutput arrays of one search as DIR/<field>.npy (integers as float64, which holds them exactly),
    so that two builds can be compared output for output on the same seeded inputs."""
    arrays = {}
    for f in DUMP_FIELDS:
        a = getattr(out, f)
        a = a.cpu().numpy() if hasattr(a, "cpu") else numpy.asarray(a)
        arrays[f] = a if a.dtype in (numpy.float32, numpy.float64) else a.astype(numpy.float64)
    assert sum(a.nbytes for a in arrays.values()) <= DUMP_MAX_BYTES
    os.makedirs(directory, exist_ok=True)
    for f, a in arrays.items():
        numpy.save(os.path.join(directory, f + ".npy"), a)


def saturation_curve(cfg, spec, N, device, dev):
    """Search throughput of the fused FC kernel at larger batches than the BASELINE's 4096 games: the headline launch
    lasts one game's chain of N dependent simulations with 28 games per SM in flight; more games per SM fill the issue
    slots that chain leaves idle (device time of 5 searches per point, inputs resident, no L2 flush)."""
    import torch
    from muzero_general_b200.engine import SearchEngine
    from muzero_general_b200.netspec import synthetic_weights
    out = []
    for B in (4096, 8192, 16384, 32768, 65536):
        eng = SearchEngine(cfg, max_games=B, device=device, num_simulations=N)
        eng.load_weights(synthetic_weights(spec, 0))
        rs = numpy.random.RandomState(B)
        obs = torch.from_numpy(rs.uniform(-0.05, 0.05, size=(B, eng.obs_elems)).astype(numpy.float32)).to(dev)
        for _ in range(2):
            eng.search(obs=obs, add_exploration_noise=True)
        ms = [eng.search(obs=obs, add_exploration_noise=True).device_ms for _ in range(5)]
        out.append({"games": B, "kernel_ms": float(numpy.median(ms)), "env_steps_per_s": B / (float(numpy.median(ms)) / 1000.0)})
        eng.close()
    return out


def selfplay_loop(game, B, N, device, rank, world, D):
    """env-steps/s of the full loop through the public API: `SelfPlay.play_moves` over B games per rank for >= 1 s."""
    from muzero_general_b200 import parallel
    from muzero_general_b200 import self_play as sp
    from muzero_general_b200.games import load_game_module
    from muzero_general_b200.netspec import netspec_from_config, synthetic_weights
    mod = load_game_module(game)
    cfg = mod.MuZeroConfig()
    cfg.num_parallel_games, cfg.rng_mode, cfg.num_simulations = B, "philox", N
    spec = netspec_from_config(cfg)
    worker = sp.SelfPlay({"weights": synthetic_weights(spec, 0)}, mod.Game, cfg, seed=0, device=device,
                         first_game_id=rank * B)
    worker.play_moves(3, 1.0)                                          # warm-up
    t0 = time.perf_counter()
    worker.play_moves(2, 1.0)
    est = D.max([(time.perf_counter() - t0) / 2])[0]
    moves = max(4, int(math.ceil(MIN_TIMED_SECONDS / max(est, 1e-9))))
    D.barrier()
    steps0, games0 = worker.env_steps, worker.played_games
    dl = getattr(worker, "_device_loop", None)
    dev0, calls0 = (dl.device_ms, dl.calls) if dl is not None else (0.0, 0)
    t0 = time.perf_counter()
    finished = worker.play_moves(moves, 1.0)
    import torch
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    lengths = [len(g.root_values) for g in finished[:64]]              # materialise a few histories: they must be real
    dt_max = D.max([dt])[0]
    table, totals = parallel.gather_counters(D.dist, worker.played_games - games0, worker.env_steps - steps0,
                                             (worker.env_steps - steps0) * N, device=torch.device("cuda", device))
    res = {"value": totals[1] / dt_max, "unit": "env-steps/s", "env_steps": int(totals[1]), "seconds": dt_max,
           "moves": moves, "games_finished": int(totals[0]), "mean_finished_length": float(numpy.mean(lengths)) if lengths else None,
           "path": worker.loop_path,
           "device_seconds": (dl.device_ms - dev0) / 1000.0 if dl is not None else None,
           "library_calls": (dl.calls - calls0) if dl is not None else None,
           "parked_events": dl.parked_events if dl is not None else None,
           "includes": "search + environment step + root noise + action sampling + GameHistory hand-over, per move"}
    worker.close()
    return res


# ----------------------------------------------------------------------------- main
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--workload", default=DEFAULT_WORKLOAD)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--extras", default=None, help="comma-separated extra workloads (name or name@tc-mode)")
    ap.add_argument("--no-extras", action="store_true")
    ap.add_argument("--no-loop", action="store_true")
    ap.add_argument("--no-saturation", action="store_true")
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the headline workload's last timed search outputs (rank 0) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.impl == "ours":
        args.warmup = max(args.warmup, 3)
    base = args.workload.partition("@")[0]
    if base not in WORKLOADS:
        raise SystemExit(f"unknown workload {args.workload}; known: {sorted(WORKLOADS)}")

    game, B, N, _ = WORKLOADS[base]
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    config = {"workload": args.workload, "game": game, "games_per_gpu": B, "num_simulations": N,
              "net": "fullyconnected" if game == "cartpole" else "resnet", "weights": "synthetic seed 0",
              "l2": "256 MiB buffer written before every timed search",
              "step": f"searches_per_step searches so that steps x step >= {MIN_TIMED_SECONDS} s",
              "value_is": "search only; loop = the whole self-play loop", "parallelism": f"games sharded x{world}"}

    # ------------------------------------------------------------------ reference arm (CPU)
    if args.impl == "reference":
        if rank != 0:
            return 0
        steps = max(1, args.steps)
        per_step = max(2.0, min(20.0, 120.0 / (steps + args.warmup)))
        arm = CpuArm(game, N)
        for _ in range(args.warmup):
            arm.run(1.0)
        total, wall = 0, 0.0
        for _ in range(steps):
            _, s, w = arm.run(per_step)
            total += s; wall += w
        arm.close()
        v = total / wall
        sample = (f"{steps} steps x {per_step:.1f}s of batch-1 MCTS.run (N={N}) on {arm.cores} processes, "
                  "one pinned per physical core")
        print(json.dumps({
            "impl": "reference", "metric": "self-play env-steps/sec", "value": v, "unit": "env-steps/s",
            "n_gpus": args.gpus, "steps": steps, "warmup": args.warmup, "ms_per_step": 1000.0 * wall / steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32+f64",
            "data": "synthetic", "config": config, "sims_per_sec": v * N,
            "cpu_baseline": {"value": v, "unit": "env-steps/s", "cores": arm.cores, "kind": "port", "sample": sample},
            "e2e": {"value": v, "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        }))
        return 0

    # ------------------------------------------------------------------ our arm (GPU)
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product path has no CPU fallback")
    dist = None
    if world > 1:
        if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
            os.environ["NCCL_DEBUG"] = "WARN"          # keep stdout to the single JSON line
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    torch.cuda.set_device(local_rank)
    D = Dist(dist, torch.device("cuda", local_rank))

    import faulthandler
    # a rank that is still here after 10 minutes writes its Python stack to stderr (and keeps going): a hung collective
    # then shows where every rank sits instead of an empty log
    faulthandler.dump_traceback_later(float(os.environ.get("MZ_BENCH_WATCHDOG", "600")), repeat=True, exit=False)

    def note(msg):
        if rank == 0:
            sys.stderr.write(f"[bench {time.strftime('%H:%M:%S')}] {msg}\n")
            sys.stderr.flush()

    note(f"{args.workload} ...")
    head = run_workload(args.workload, args, D, rank, local_rank, world, with_loop=not args.no_loop, headline=True)
    note(f"{args.workload}: {head['value']:.0f} env-steps/s, loop {(head.get('loop') or {}).get('value')}")
    extras = {}
    names = [] if args.no_extras else (args.extras.split(",") if args.extras else DEFAULT_EXTRAS)
    for nme in names:
        if not nme or nme == args.workload:
            continue
        try:
            note(f"{nme} ...")
            extras[nme] = run_workload(nme, args, D, rank, local_rank, world,
                                       with_loop=(not args.no_loop and "@" not in nme), headline=False)
        except Exception as e:
            if world > 1:
                raise                                   # a rank that skips its collectives would hang the others
            extras[nme] = {"error": repr(e)}

    if rank == 0:
        out = {
            "metric": "self-play env-steps/sec", "value": head["value"], "unit": "env-steps/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": head["ms_per_step"],
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": head["dtype"], "data": "synthetic", "config": dict(config, searches_per_step=head["searches_per_step"]),
            "sims_per_sec": head["sims_per_sec"], "ms_per_search": head["ms_per_search"],
            "kernel_ms_per_search": head["kernel_ms_per_search"], "timed_seconds": head["timed_seconds"],
            "e2e": head["e2e"], "gpu_launches": head["gpu_launches"], "clocks": head.get("clocks"),
            "roofline": head["roofline"],
        }
        if "loop" in head:
            out["loop"] = head["loop"]
        if "saturation" in head:
            out["saturation"] = head["saturation"]
        if extras:
            out["workloads"] = extras
        if world == 1 and not args.no_cpu_baseline:
            arm = CpuArm(game, N)
            v, searches, w = arm.run(args.cpu_seconds)
            arm.close()
            out["cpu_baseline"] = {"value": v, "unit": "env-steps/s", "cores": arm.cores, "kind": "port",
                                   "sample": f"{searches} batch-1 MCTS.run calls (N={N}) in {w:.1f}s on {arm.cores} processes, "
                                             "one pinned per physical core"}
        print(json.dumps(out))
    faulthandler.cancel_dump_traceback_later()
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
