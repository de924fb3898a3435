#!/usr/bin/env python
"""bench.py -- Azul env steps/s of the batched random-agent rollout (BASELINE.json configs[1]) and, in the same JSON
line, the other configurations of SURVEY.md §8(d).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--mode random|step|config3|policy|train]
                    [--dump-outputs DIR]

Headline (mode "random", the default): one bench "step" = ONE launch of the fused rollout kernel (azb_rollout_random:
legal mask + random agent + Azul.step + scoring + refill + auto-reset) that advances every one of the G games by
--k-steps env steps.  N = 1 runs BASELINE.json configs[1] (65,536 parallel 2-player random-agent games); N > 1
(torchrun, one rank per GPU) shards the global game-id range over the ranks with no data-path collective (weak
scaling, G games per GPU); NCCL carries the max-over-ranks timing, the rollout-counter reduction and -- in the
training extra -- the gradient all-reduce.

The JSON line carries
  value      env steps/s, state resident in HBM, timed with CUDA events on the launching stream
  e2e        the same metric through the public host API with HOST buffers: per step the packed state is copied from
             pinned host memory to the device, rolled out, and state + legal mask + counters are copied back
  roofline   algorithmic bytes (BASELINE.md §4: 2*S(P)+25 per env step) / kernel time vs the measured HBM peak, plus
             issue_frac: the kernel's warp instructions per env step (ncu) against the SMs' issue rate at the sampled clock
  cpu_baseline  the C oracle port (kind "port") on all host threads on a bounded sample, and python_reference: the
             UNMODIFIED reference's GameRunner loop (baseline/_ref, copied by build()) on os.cpu_count() processes
  extra      step (azb_step, the HBM-bound single-step entry point, 4.2 M games), config3 (P = 2, 3, 4 at 262,144 games
             per GPU), policy (configs[3]: fused tcgen05 policy kernel self-play) and train (configs[4]: rollouts + A2C
             update + gradient all-reduce), each measured like the headline with its own clocks and roofline
--impl reference times the reference arm for this tier: the oracle port on all host threads, same config / metric / unit.
--dump-outputs DIR writes what the measured path (the headline, or the --mode) returned in its last timed step: random and
config3: state (packed words [W, G]), legal_mask ([6, G]), counters; step: state, legal_mask, done, status; policy: state,
counters; train: the network's parameters (param.*) and the last batch's statistics (stat.*).  The inputs are seeded, so
two builds run with the same arguments can be compared file by file.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

REPO = os.path.dirname(os.path.abspath(__file__))
if REPO not in sys.path:
    sys.path.insert(0, REPO)

METRIC = "azul_env_steps_per_sec"
UNIT = "env_steps/s"
FALLBACK_HBM_GBS = 6650.0          # /opt/skills/guides/B200_PROFILING.md fallback
PYREF_DIR = os.path.join(REPO, "baseline", "_ref")     # unmodified reference, copied by __graft_entry__.build()


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--mode", default="random", choices=["random", "policy", "train", "step", "config3"],
                    help="random: fused random-agent rollout (configs[1], the headline, with the other modes as `extra`); "
                         "step: azb_step; config3: P = 2,3,4 at 262,144 games; policy: fused policy kernel self-play "
                         "(configs[3]); train: self-play A2C training (configs[4])")
    ap.add_argument("--games", type=int, default=0, help="games per GPU (default 65536 random / 131072 policy / 16384 train / 4194304 step)")
    ap.add_argument("--players", type=int, default=2)
    ap.add_argument("--pool", default="lid", choices=["lid", "random"],
                    help="tile pool; 'lid' + random first player = GameRunner's default rules (game_runner.py:23)")
    ap.add_argument("--k-steps", type=int, default=4096,
                    help="env steps per game per launch (SURVEY §8d config 2: K = 4,096 with auto-reset)")
    ap.add_argument("--block", type=int, default=0, help="threads per block (0 = library default)")
    ap.add_argument("--defer", type=int, default=0, help="rollout end-of-round batching threshold (0 = library default)")
    ap.add_argument("--seed", type=lambda s: int(s, 0), default=0x5EED)
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="target CPU time of the cpu_baseline sample (C port)")
    ap.add_argument("--pyref-seconds", type=float, default=20.0,
                    help="wall time of the Python-reference leg (BASELINE.md §3: >= 20 s); 0 skips it")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="headline only (no step / config3 / policy / train extras)")
    ap.add_argument("--step-actions", default="random", choices=["random", "lowest"],
                    help="--mode step: the caller-supplied action per game (a random or the lowest legal one)")
    ap.add_argument("--presteps", type=int, default=203,
                    help="--mode step: random-agent env steps before the timed step (0 = fresh games: no round can end)")
    ap.add_argument("--policy-k", type=int, default=64, help="policy: decisions per game per launch of the persistent self-play kernel")
    ap.add_argument("--no-graph", action="store_true", help="train: run the batch launch by launch instead of as one CUDA graph")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the measured path returned in its last step as DIR/<name>.npy "
                         "(integers as float64, floating point as float32; rank 0's games; at most 64 MB, a fixed sample "
                         "of the games beyond that)")
    ap.add_argument("--pyref-worker", type=float, default=None, help=argparse.SUPPRESS)
    ap.add_argument("--pyref-kind", default="runner", choices=["runner", "selfplay", "train"], help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the CUDA path (--impl b200)")
    return args


def workload_config(args, n_gpus, games=None, players=None):
    games = args.games if games is None else games
    players = args.players if players is None else players
    return {
        "workload": "%d parallel %d-player random-agent Azul games per GPU, env step + legal mask, auto-reset "
                    "(BASELINE.json configs[1])" % (games, players),
        "games_per_gpu": games, "players": players,
        "rules": {"tile_pool": "Lid" if args.pool == "lid" else "Random", "first_player": "Random"},
        "env_steps_per_game_per_launch": args.k_steps,
        "rng": "Philox4x32-10, seed 0x%X, keyed by global game id" % args.seed,
        "l2": "flushed between timed launches (256 MiB device fill outside the CUDA-event brackets)",
        "parallelism": "games sharded by global id over %d GPU(s); no data-path collective" % n_gpus,
    }


# ------------------------------------------------------------------------------------------
# CPU legs: the C oracle port (cpu_baseline / --impl reference) and the unmodified Python reference
# ------------------------------------------------------------------------------------------
def cpu_rollout_rate(args, seconds, threads):
    """Time the C oracle's rollout (same Philox schedule, same rules) on `threads` host threads."""
    from oracle import oracle as O
    pool = 1 if args.pool == "lid" else 0
    probe_n, probe_k = 256 * threads, 64
    recs = O.fresh_records(probe_n, args.players, pool, 0, args.seed, 0)
    t0 = time.perf_counter()
    O.rollout_random(recs, args.players, pool, 0, args.seed, 0, probe_k, threads=threads)
    rate = probe_n * probe_k / max(time.perf_counter() - t0, 1e-6)
    k = args.k_steps
    n = int(max(threads, min(args.games, rate * seconds / k)))
    recs = O.fresh_records(n, args.players, pool, 0, args.seed, 0)
    t0 = time.perf_counter()
    cnt = O.rollout_random(recs, args.players, pool, 0, args.seed, 0, k, threads=threads)
    dt = time.perf_counter() - t0
    assert cnt[0] == n * k
    return n * k / dt, n, k, dt


def cpu_model_name():
    try:
        for ln in open("/proc/cpuinfo"):
            if ln.lower().startswith("model name"):
                return ln.split(":", 1)[1].strip()
    except OSError:
        pass
    return "unknown"


def pyref_worker(seconds, kind="runner"):
    """One process of the Python-reference leg, on the UNMODIFIED reference (baseline/_ref):
    runner    GameRunner (game_runner.py:9-85, default rules), seat 1 driven by its RandomAgent against its RandomAgent
              opponent (BASELINE.json configs[0])
    selfplay  NNRunner.run_episode (nn_runner.py:17-47) of a random-init Agent against a random-init Agent opponent
              (scripts/run_batch.py: every seat sampled from the policy, configs[3])
    train     NNRunner.train(batch_size=10, batches=1) (scripts/training.py defaults, configs[4])"""
    sys.path.insert(0, PYREF_DIR)
    import numpy as np
    if not hasattr(np, "int"):
        np.int = int              # removed in numpy 1.24; azul.py:19 (the only shim; the sources are untouched)
    if not hasattr(np, "bool"):
        np.bool = bool
    import random
    import torch
    torch.set_num_threads(1)
    from azulnet.game_runner import GameRunner, RandomAgent
    if kind == "runner":
        agent, gr = RandomAgent(), GameRunner()

        def episode(seed):
            random.seed(seed)
            gr.reset()
            done = False
            while not done:
                valid = gr.get_valid_moves()
                a = agent.get_a_output(None, torch.from_numpy(valid.reshape(1, 180)))
                _, done = gr.step(a)
            return gr.move_counter, 1
    else:
        from azulnet.agent import Agent
        from azulnet.nn_runner import NNRunner
        torch.manual_seed(0)
        learner = Agent()
        gr = GameRunner(opponent=Agent()) if kind == "selfplay" else GameRunner()
        runner = NNRunner(learner, gr)
        counted = {"steps": 0}

        def episode(seed):
            import numpy
            random.seed(seed)
            numpy.random.seed(seed % (2 ** 31))
            if kind == "selfplay":
                runner.run_episode()
                return gr.move_counter, 1
            n0 = counted["steps"]
            orig_reset = gr.reset

            def reset():                                  # GameRunner.reset zeroes move_counter: bank the finished episode first
                counted["steps"] += gr.move_counter
                orig_reset()
            gr.reset = reset
            try:
                runner.train(net_name=None, batch_size=10, batches=1)
            finally:
                gr.reset = orig_reset
            counted["steps"] += gr.move_counter
            gr.move_counter = 0
            return counted["steps"] - n0, 10

    seed = os.getpid() * 1000
    episode(seed)                                     # warm-up
    print("ready", flush=True)
    sys.stdin.readline()                              # the parent releases all workers together
    steps = games = crashed = 0
    t0 = time.perf_counter()
    while time.perf_counter() - t0 < seconds:
        seed += 1
        try:
            st, n = episode(seed)
            steps += st
            games += n
        except (ValueError, IndexError):              # stuck round: the reference crashes (SURVEY §5); not counted
            crashed += 1
    print(json.dumps({"steps": steps, "games": games, "seconds": time.perf_counter() - t0, "crashed": crashed}), flush=True)


def _run_pyref_workers(n, seconds, kind="runner"):
    procs = [subprocess.Popen([sys.executable, os.path.abspath(__file__), "--pyref-worker", str(seconds), "--pyref-kind", kind],
                              stdin=subprocess.PIPE, stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, cwd=REPO)
             for _ in range(n)]
    try:
        for p in procs:
            if p.stdout.readline().strip() != "ready":
                raise RuntimeError("python-reference worker failed to start")
        for p in procs:
            p.stdin.write("go\n")
            p.stdin.flush()
        res = [json.loads(p.stdout.readline()) for p in procs]
    finally:
        for p in procs:
            try:
                p.stdin.close()
            except Exception:
                pass
            p.wait(timeout=60)
    wall = max(r["seconds"] for r in res)
    return sum(r["steps"] for r in res), sum(r["games"] for r in res), wall, sum(r["crashed"] for r in res)


PYREF_WHAT = {
    "runner": "unmodified azulnet GameRunner (default rules: random first player, Lid pool), RandomAgent on both seats (BASELINE.json configs[0])",
    "selfplay": "unmodified azulnet NNRunner.run_episode, random-init Agent against a random-init Agent opponent (scripts/run_batch.py; configs[3] on the CPU)",
    "train": "unmodified azulnet NNRunner.train(batch_size=10, batches=1) per iteration, Agent vs RandomAgent (scripts/training.py; configs[4] on the CPU)",
}


def python_reference_leg(seconds, kind="runner"):
    """BASELINE.md §3: the reference CPU game_runner on this host, os.cpu_count() single-threaded processes for
    `seconds` of wall time after warm-up, plus the single-core figure (one process alone)."""
    if seconds <= 0:
        return None
    if not os.path.isfile(os.path.join(PYREF_DIR, "azulnet", "game_runner.py")):
        return {"unavailable": "baseline/_ref not present (build() copies it from /root/reference when that exists)"}
    cores = os.cpu_count() or 1
    try:
        s1, g1, w1, _ = _run_pyref_workers(1, min(5.0, seconds), kind)
        s, g, w, crashed = _run_pyref_workers(cores, seconds, kind)
    except Exception as e:            # never let the reported baseline take the GPU numbers down
        return {"unavailable": "python reference leg failed: %s" % e}
    return {"value": s / w, "unit": UNIT, "games_per_sec": g / w, "cores": cores, "cpu_model": cpu_model_name(),
            "kind": "reference", "single_core_value": s1 / w1, "single_core_games_per_sec": g1 / w1,
            "env_steps": s, "games": g, "wall_s": w, "episodes_crashed": crashed,
            "sample": "%s; %d single-threaded processes x %.0f s wall after warm-up; %d games, %d env steps" % (
                PYREF_WHAT[kind], cores, w, g, s)}


def run_reference_python(args, kind):
    """--impl reference for the modes whose path includes the MLP (policy, train): there is no C port of those; the arm is
    the unmodified Python reference itself on all host cores."""
    py = python_reference_leg(max(args.pyref_seconds, 5.0), kind)
    cfg = workload_config(args, args.gpus)
    cfg["workload"] = PYREF_WHAT[kind]
    cfg.pop("env_steps_per_game_per_launch", None)
    if py is None or "unavailable" in py:
        print(json.dumps({"impl": "reference", "unavailable": (py or {}).get("unavailable", "python reference leg disabled")}))
        return
    line = {"impl": "reference", "metric": METRIC, "value": py["value"], "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * py["wall_s"] / max(args.steps, 1), "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "fp32 (torch CPU) / python int", "data": "synthetic", "config": cfg,
            "cpu_baseline": dict(py), "games_per_sec": py["games_per_sec"],
            "e2e": {"value": py["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return                                   # rank 0 alone runs the CPU arm
    if args.mode in ("policy", "train"):
        return run_reference_python(args, "selfplay" if args.mode == "policy" else "train")
    threads = os.cpu_count() or 1
    pool = 1 if args.pool == "lid" else 0
    from oracle import oracle as O
    # bounded sample per step so the whole run ends within minutes: ~0.5 s of CPU work per step
    rate, _, _, _ = cpu_rollout_rate(args, 1.0, threads)
    n = int(max(threads, min(args.games, rate * 0.5 / args.k_steps)))
    recs = O.fresh_records(n, args.players, pool, 0, args.seed, 0)
    for _ in range(args.warmup):
        O.rollout_random(recs, args.players, pool, 0, args.seed, 0, args.k_steps, threads=threads)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        O.rollout_random(recs, args.players, pool, 0, args.seed, 0, args.k_steps, threads=threads)
    dt = time.perf_counter() - t0
    value = n * args.k_steps * args.steps / dt
    sample = ("%d of %d games x %d env steps per step (bounded sample: the rate does not depend on the batch size), "
              "C oracle port (oracle/azul_oracle.c), %d threads" % (n, args.games, args.k_steps, threads))
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u32", "data": "synthetic",
        "config": workload_config(args, args.gpus),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample,
                         "cpu_model": cpu_model_name()},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "note": "this arm is the C restatement of the reference's rules, pinned bit-exactly to the unmodified reference "
                "(tests/test_oracle_golden.py, tests/test_runner_golden_cpu.py), on all host threads; "
                "cpu_baseline.python_reference is the unmodified Python reference itself (baseline/_ref) on the same cores.",
    }
    py = python_reference_leg(args.pyref_seconds)
    if py is not None:
        line["cpu_baseline"]["python_reference"] = py
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------
# clocks
# ------------------------------------------------------------------------------------------
class ClockSampler:
    """SM clock + throttle reasons sampled every 10 ms through NVML (nvidia_ml_py) while the timed region
    runs; falls back to an `nvidia-smi -lms` subprocess (the profiling recipe's clocks line)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")
    REASONS = {0x4: "sw_power_cap", 0x8: "hw_slowdown", 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown",
               0x80: "hw_power_brake_slowdown"}

    def __init__(self, torch_device_index):
        import threading
        self.idx, self.proc, self.thread, self.stop_flag = torch_device_index, None, None, threading.Event()
        self.sm, self.bits, self.max_mhz, self.power = [], 0, None, []
        self.nvml = None
        try:
            import pynvml
            import torch
            pynvml.nvmlInit()
            try:
                uuid = "GPU-" + str(torch.cuda.get_device_properties(torch_device_index).uuid)
                self.h = pynvml.nvmlDeviceGetHandleByUUID(uuid)
            except Exception:
                self.h = pynvml.nvmlDeviceGetHandleByIndex(torch_device_index)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.nvml = pynvml
        except Exception:
            self.nvml = None

    def _loop(self):
        nv = self.nvml
        while not self.stop_flag.is_set():
            try:
                self.sm.append(float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                self.bits |= int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
                self.power.append(nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0)
            except Exception:
                pass
            self.stop_flag.wait(0.01)

    def start(self):
        if self.nvml is not None:
            import threading
            self.thread = threading.Thread(target=self._loop, daemon=True)
            self.thread.start()
            return
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                 "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            self.proc = None

    def stop(self):
        if self.thread is not None:
            self.stop_flag.set()
            self.thread.join()
            reasons = sorted(name for bit, name in self.REASONS.items() if self.bits & bit)
            return {"sm_mhz": statistics.median(self.sm) if self.sm else None, "sm_max_mhz": self.max_mhz,
                    "samples": len(self.sm), "power_w_max": max(self.power) if self.power else None,
                    "reasons": reasons, "source": "nvml, 10 ms period, timed region only"}
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no clock source available"]}
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
            out, _ = self.proc.communicate()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in out.strip().splitlines():
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons), "source": "nvidia-smi -lms 100"}


# ------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------
def measured_peaks():
    try:
        return json.load(open(os.path.join(REPO, "MEASURED_PEAKS.json")))
    except Exception:
        return {}


def hbm_peak():
    p = measured_peaks()
    if "hbm_gbs" in p:
        return float(p["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return FALLBACK_HBM_GBS, "fallback (B200_PROFILING.md 6.65 TB/s)"


def profiled(key):
    """Per-launch figures taken from the committed ncu captures (profiles/rollout_traffic.json), or None."""
    try:
        return json.load(open(os.path.join(REPO, "profiles", "rollout_traffic.json"))).get(key)
    except Exception:
        return None


class Ctx:
    """Rank / device plumbing shared by the measurements of one bench process."""

    def __init__(self, args):
        import torch
        from azul_deep_reinforcement_learning_b200 import parallel
        self.torch, self.parallel = torch, parallel
        self.rank, self.world, self.local = parallel.world()
        if self.world > 1:
            parallel.init("nccl", self.local)
        assert self.world == args.gpus or self.world == 1, "launch with torchrun --nproc-per-node %d" % args.gpus
        torch.cuda.set_device(self.local)
        self.dev = torch.device("cuda", self.local)
        self.pool = 1 if args.pool == "lid" else 0
        self._flush = None

    def barrier(self):
        if self.world > 1:
            self.torch.distributed.barrier()
        self.torch.cuda.synchronize()

    def flush_l2(self, tag=0):
        if self._flush is None:
            self._flush = self.torch.empty(256 << 20, dtype=self.torch.uint8, device=self.dev)
        self._flush.fill_(tag & 0xFF)

    def max_over_ranks(self, v):
        return self.parallel.max_over_ranks(v, self.dev)

    def clocks(self):
        return ClockSampler(self.local)

    def close(self):
        if self.world > 1:
            self.torch.distributed.destroy_process_group()


def rollout_kernel_name(games, players, pool, sms, tuned):
    """Which kernel azb_rollout_random picks (csrc/azb.cu): one block per SM whose 32-game batches number 2 mod 4 (65,536 games
    on 148 SMs: 14) -> the rotating form, two warps more than batches; otherwise one warp per batch for the whole launch."""
    per_sm = -(-games // sms)
    k = -(-per_sm // 512)
    threads = min(512, max(64, -(-(-(-per_sm // k)) // 32) * 32))
    rotate = (not tuned and per_sm <= 2048 and (threads // 32) % 4 == 2 and threads + 64 <= 512 and -(-games // threads) <= sms)
    return ("k_rollout_rotate<%d,%d>" if rotate else "k_rollout_random<%d,%d>") % (players, pool)


def measure_random(args, ctx, players, games, steps, warmup, e2e=True):
    """configs[1] / configs[2]: azb_rollout_random, K env steps per game per launch, L2 flushed between launches."""
    torch = ctx.torch
    from azul_deep_reinforcement_learning_b200.engine import BatchedAzul
    from azul_deep_reinforcement_learning_b200.layout import algorithmic_bytes_per_step
    G, K, world = games, args.k_steps, ctx.world
    eng = BatchedAzul(G, players, ctx.pool, 0, seed=args.seed, device=ctx.local, game_id_base=ctx.parallel.shard(ctx.rank, G))
    if args.block:
        eng.set_block_threads(args.block)
    if args.defer:
        eng.set_rollout_defer(args.defer)
    mask = torch.empty((6, G), dtype=torch.int32, device=ctx.dev)
    for _ in range(warmup):
        eng.rollout_random(K, mask)
    ctx.barrier()
    sampler = ctx.clocks()
    if ctx.rank == 0:
        sampler.start()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    ctx.barrier()
    t_wall0 = time.perf_counter()
    for s in range(steps):
        ctx.flush_l2(s)                          # L2 flush, outside the event bracket
        ev[s][0].record()
        eng.rollout_random(K, mask)
        ev[s][1].record()
    ctx.barrier()
    wall = time.perf_counter() - t_wall0
    clocks = sampler.stop() if ctx.rank == 0 else None
    kernel_ms = [a.elapsed_time(b) for a, b in ev]
    dev_ms = sum(kernel_ms)
    dev_ms_max = ctx.max_over_ranks(dev_ms)
    outputs = None
    if args.dump_outputs:                        # copied now: the e2e leg below rolls the same engine on
        outputs = ({"state": eng.state.clone(), "legal_mask": mask.clone()}, {"counters": eng.counters.clone()})
    out_e2e = None
    if e2e:
        # ---- end to end through the host API ----
        host_state = torch.empty(eng.state.shape, dtype=torch.int32).pin_memory()
        host_state.copy_(eng.state)
        host_mask = torch.empty((6, G), dtype=torch.int32).pin_memory()
        host_cnt = torch.empty(16, dtype=torch.int64).pin_memory()
        e2e_steps = max(3, min(steps, 10))
        for _ in range(2):
            eng.rollout_random_host(host_state, K, host_mask, host_cnt)
        ctx.barrier()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            eng.rollout_random_host(host_state, K, host_mask, host_cnt)
        ctx.barrier()
        e2e_s = ctx.max_over_ranks(time.perf_counter() - t0)
        out_e2e = {"value": world * G * K * e2e_steps / e2e_s, "unit": UNIT, "h2d_bytes_per_step": host_state.numel() * 4,
                   "d2h_bytes_per_step": host_state.numel() * 4 + host_mask.numel() * 4 + host_cnt.numel() * 8,
                   "steps": e2e_steps}
    cnt = ctx.parallel.reduce_counters(eng.counters.clone()).cpu().tolist()      # C2: one small all-reduce
    value = world * G * K * steps / (dev_ms_max * 1e-3)
    b_alg = algorithmic_bytes_per_step(players)
    achieved = b_alg * G * K / ((dev_ms / steps) * 1e-3) / 1e9
    peak, peak_src = hbm_peak()
    pool_name = "lid" if ctx.pool else "random"
    kernel_name = rollout_kernel_name(G, players, ctx.pool, torch.cuda.get_device_properties(ctx.dev).multi_processor_count,
                                      bool(args.block or args.defer))
    rot = "_rotate" if "rotate" in kernel_name else ""
    inst = (profiled("inst_per_env_step_p%d_%s%s" % (players, pool_name, rot)) or profiled("inst_per_env_step_p2_lid" + rot)
            or profiled("inst_per_env_step_p2_lid"))
    roof = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
            "traffic": profiled("p%d_%s_g%d_k%d%s" % (players, pool_name, G, K, rot)) or profiled("p%d_%s_g%d_k%d" % (players, pool_name, G, K)),
            "peak_source": peak_src,
            "algorithmic_bytes_per_env_step": b_alg, "env_steps_per_launch": G * K,
            "kernel": kernel_name,
            "kernel_ms_avg": dev_ms / steps, "kernel_ms_min": min(kernel_ms)}
    # frac follows the metric's definition (algorithmic bytes of a step-at-a-time simulator / time / measured copy peak); the fused
    # kernel keeps the state in registers for K steps, so the figure is not bounded by 1 -- `traffic` is what DRAM really moved
    roof["frac_note"] = ("algorithmic bytes per SURVEY 8(d) (2*S(P)+25 per env step) over the measured HBM copy peak; the K-step kernel "
                         "keeps the state in registers (DRAM traffic per launch = `traffic`), so frac can exceed 1: the physical "
                         "bound is instruction issue (issue_frac)")
    if inst and clocks and clocks.get("sm_mhz"):
        # the physical bound of this kernel (state lives in registers for K steps: DRAM traffic is ~1e-4 of the algorithmic
        # bytes): warp instructions per env step (ncu, profiles/) against sm_count x 4 schedulers x 1 instruction / cycle
        sms = torch.cuda.get_device_properties(ctx.dev).multi_processor_count
        issue_peak = sms * 4 * clocks["sm_mhz"] * 1e6 / inst
        roof.update(issue_frac=(value / world) / issue_peak, issue_peak_env_steps_per_sec=issue_peak,
                    warp_instructions_per_env_step=inst,
                    issue_note="warp instructions per env step from the committed ncu capture; peak = SMs x 4 x sampled SM clock / that")
    alu = profiled("alu_pipe_pct_p%d_%s_g%d%s" % (players, pool_name, G, rot))
    if alu:
        roof.update(alu_pipe_busy_pct_ncu=alu,
                    alu_note="integer ALU pipe utilisation of this kernel at this batch size in the committed ncu capture "
                             "(profiles/rollout_traffic.json): the unit closest to its peak, i.e. the kernel's binding pipe")
    return {"value": value, "unit": UNIT, "n_gpus": world, "steps": steps, "warmup": warmup,
            "ms_per_step": dev_ms_max / steps, "e2e": out_e2e, "gpu_launches": steps, "roofline": roof, "clocks": clocks,
            "wall_s": wall, "games_per_sec": (cnt[1] / max(cnt[0], 1)) * value,
            "rollout_counters": {"steps": cnt[0], "games": cnt[1], "rounds": cnt[2], "stuck": cnt[6]},
            "config": workload_config(args, world, games=G, players=players), "outputs": outputs}


def measure_step(args, ctx, games, players, steps, warmup):
    """The single-step entry point the reference's callers use (one Azul.step + next legal mask per call, actions
    supplied by the caller): a genuinely HBM-bound pass -- packed state read + written, 1 action byte in, 24 mask bytes
    + done + status out per game -- on a batch larger than L2."""
    import ctypes
    torch = ctx.torch
    from azul_deep_reinforcement_learning_b200.engine import BatchedAzul, mask_to_bool
    from azul_deep_reinforcement_learning_b200.layout import algorithmic_bytes_per_step
    G, dev = games, ctx.dev
    eng = BatchedAzul(G, players, ctx.pool, 0, seed=args.seed, device=ctx.local, game_id_base=ctx.parallel.shard(ctx.rank, G))
    eng.rollout_random(args.presteps)
    mask = eng.legal_mask()
    done = torch.empty(G, dtype=torch.uint8, device=dev)
    status = torch.empty(G, dtype=torch.uint8, device=dev)
    # one legal action per game, computed once outside the timing: uniformly random among the legal ones (default: the
    # share of games whose round ends in the timed step is then that of random play, ~1 in 10) or the lowest one
    action = torch.empty(G, dtype=torch.uint8, device=dev)
    gen = torch.Generator(device=dev).manual_seed(args.seed + ctx.rank)
    for lo in range(0, G, 1 << 20):                   # chunked: the bool [G, 180] expansion of 4.2 M masks is 755 MB
        legal = mask_to_bool(mask[:, lo:lo + (1 << 20)])
        if args.step_actions == "random":
            action[lo:lo + (1 << 20)] = torch.multinomial(legal.float() + 1e-12, 1, generator=gen).squeeze(1).to(torch.uint8)
        else:
            action[lo:lo + (1 << 20)] = legal.to(torch.uint8).argmax(dim=1).to(torch.uint8)
        del legal
    snapshot = eng.state.clone()
    st = ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    p = lambda t: ctypes.c_void_p(t.data_ptr())   # noqa: E731

    def launch():
        assert eng.lib.azb_step(eng._h, p(eng.state), p(action), None, p(mask), None, p(done), p(status), st) == 0

    ms = []
    sampler = ctx.clocks()
    ctx.barrier()
    for i in range(warmup + steps):
        if i == warmup and ctx.rank == 0:
            sampler.start()
        eng.state.copy_(snapshot)                 # same legal actions every iteration; the 285 MB copy also turns L2 over
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); launch(); e1.record()
        torch.cuda.synchronize()
        if i >= warmup:
            ms.append(e0.elapsed_time(e1))
    clocks = sampler.stop() if ctx.rank == 0 else None
    ctx.barrier()
    assert int(status.max()) & 3 == 0
    # MISC word: turn_counter [27:16] moves on new_round, end_of_game [12] when the scored round finished the game
    round_ends = float((((eng.state[3] ^ snapshot[3]) & ((0xFFF << 16) | (1 << 12))) != 0).float().mean())
    b_alg = algorithmic_bytes_per_step(players) + 2
    t = ctx.max_over_ranks(statistics.median(ms)) * 1e-3
    peak, src = hbm_peak()
    pool_name = "lid" if ctx.pool else "random"
    cfg = workload_config(args, ctx.world, games=G, players=players)
    cfg["workload"] = "%d parallel %d-player games per GPU, ONE Azul.step + next legal mask per launch, caller-supplied actions (azb_step)" % (G, players)
    cfg["env_steps_per_game_per_launch"] = 1
    cfg["actions"] = "%s legal action per game after %d random-agent steps; %.1f %% of the games end their round (score + refill) in the timed step" % (
        args.step_actions, args.presteps, 100 * round_ends)
    cfg["l2"] = "working set %.0f MB per launch (state %d B + 28 B per game) exceeds the 126 MB L2; the state is restored from a snapshot before every launch" % (G * b_alg / 1e6, 4 * eng.W)
    outputs = ({"state": eng.state, "legal_mask": mask, "done": done, "status": status}, {}) if args.dump_outputs else None
    return {"value": ctx.world * G / t, "unit": UNIT, "n_gpus": ctx.world, "steps": steps, "warmup": warmup, "ms_per_step": 1e3 * t,
            "dtype": "u32", "config": cfg, "gpu_launches": steps, "clocks": clocks, "outputs": outputs,
            "roofline": {"bound": "hbm", "achieved": G * b_alg / t / 1e9, "peak": peak, "unit": "GB/s",
                         "frac": G * b_alg / t / 1e9 / peak,
                         "traffic": profiled("step_p%d_%s_g%d_%s" % (players, pool_name, G, args.step_actions)),
                         "peak_source": src, "algorithmic_bytes_per_env_step": b_alg, "kernel": "k_step<%d,%d>" % (players, ctx.pool),
                         "kernel_ms_median": 1e3 * t, "kernel_ms_min": min(ms)}}


def policy_accuracy(eng, packed, net, G):
    """SURVEY §8(d) config 4: logits / value of the kernel (fp16 operands, fp32 accumulation) against the untouched fp32
    ActorCritic forward (model.py:23-41) on the CPU, 4,096 of the mid-game states reached by the bench; outside the timing."""
    import torch
    from azul_deep_reinforcement_learning_b200.engine import policy_step
    with torch.no_grad():
        chk = policy_step(eng, packed, mode=1, apply_step=False, want_logits=True, want_mask=False)
        k = min(4096, G)
        obs = eng.observe(-1)[:k].cpu()
        ref_l = net.actor_linear2(torch.relu(net.actor_linear1(obs)))
        ref_v = net.forward_critic(obs).squeeze(1)
        got_l, got_v = chk["logits"][:k].cpu(), chk["value"][:k].cpu()
        err = (got_l - ref_l).abs()
        row = ref_l.abs().max(dim=1, keepdim=True).values
        return {"states": k, "reference": "fp32 ActorCritic forward on the CPU (torch)",
                "logits_max_abs_err": float(err.max()), "logits_mean_abs_err": float(err.mean()),
                "logits_max_abs": float(ref_l.abs().max()),
                "logits_max_err_rel_to_scale": float(err.max() / ref_l.abs().max()),
                "logits_max_err_rel_to_row_max": float((err / row).max()),
                "value_max_abs_err": float((got_v - ref_v).abs().max())}


def measure_policy(args, ctx, games, steps, warmup):
    """BASELINE.json configs[3]: self-play, every seat sampled from a random-init ActorCritic (model.py:17-21 under
    torch.manual_seed(0)) by the fused policy kernel.  One bench step = ONE launch of the persistent self-play kernel
    (azb_policy_rollout): --policy-k decisions (= env steps) per game, state resident on the device in between."""
    torch = ctx.torch
    from azul_deep_reinforcement_learning_b200.azulnet.model import ActorCritic
    from azul_deep_reinforcement_learning_b200.engine import BatchedAzul, PackedPolicy
    G, world, dev, K = games, ctx.world, ctx.dev, args.policy_k
    torch.manual_seed(0)
    net = ActorCritic(136, 180)
    eng = BatchedAzul(G, 2, ctx.pool, 0, seed=args.seed, device=ctx.local, game_id_base=ctx.parallel.shard(ctx.rank, G))
    packed = PackedPolicy(eng, net)
    for _ in range(warmup + 1):                      # warm-up also spreads the games over all phases of a game
        eng.policy_rollout(packed, K)
    ctx.barrier()
    sampler = ctx.clocks()
    if ctx.rank == 0:
        sampler.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ctx.barrier()
    ev0.record()
    for _ in range(steps):
        eng.policy_rollout(packed, K)
    ev1.record()
    ctx.barrier()
    clocks = sampler.stop() if ctx.rank == 0 else None
    dev_ms = ctx.max_over_ranks(ev0.elapsed_time(ev1))
    outputs = None
    if args.dump_outputs:                        # copied now: the e2e leg below plays the same games on
        outputs = ({"state": eng.state.clone()}, {"counters": eng.counters.clone()})
    # end to end: pinned host state in, K decisions per game, state + the last decision's action / logp / value + counters out
    host_state = torch.empty(eng.state.shape, dtype=torch.int32).pin_memory()
    host_state.copy_(eng.state)
    host_last = {"action": torch.empty(G, dtype=torch.uint8).pin_memory(), "logp": torch.empty(G, dtype=torch.float32).pin_memory(),
                 "value": torch.empty(G, dtype=torch.float32).pin_memory()}
    host_cnt = torch.empty(16, dtype=torch.int64).pin_memory()
    e2e_steps = max(3, min(steps, 10))
    eng.policy_rollout_host(packed, host_state, K, host_last, host_cnt)
    ctx.barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        eng.policy_rollout_host(packed, host_state, K, host_last, host_cnt)
    ctx.barrier()
    e2e_s = ctx.max_over_ranks(time.perf_counter() - t0)
    cnt = ctx.parallel.reduce_counters(eng.counters.clone()).cpu().tolist()
    accuracy = policy_accuracy(eng, packed, net, G) if ctx.rank == 0 else None
    value = world * G * K * steps / (dev_ms * 1e-3)
    flop = 2 * (136 * 360 + 180 * 180 + 180)                                  # SURVEY §8d: 163,080 per decision
    peaks = measured_peaks()
    peak = float(peaks.get("bf16_tflops", 1590.0))
    achieved = flop * (value / world) / 1e12
    cfg = workload_config(args, world, games=G, players=2)
    cfg["workload"] = ("%d parallel 2-player self-play games per GPU, every seat sampled from a random-init "
                       "ActorCritic(136,180) by the fused policy kernel (BASELINE.json configs[3])" % G)
    cfg["env_steps_per_game_per_launch"] = K
    cfg["l2"] = "working set (%.1f MB packed state) stays resident across the %d decisions of a launch; no flush" % (eng.state.numel() * 4 / 1e6, K)
    return {"value": value, "unit": UNIT, "n_gpus": world, "steps": steps, "warmup": warmup + 1,
            "ms_per_step": dev_ms / steps, "dtype": "fp16 operands, fp32 accumulate (MLP) / u32 (rules)", "config": cfg,
            "e2e": {"value": world * G * K * e2e_steps / e2e_s, "unit": UNIT, "h2d_bytes_per_step": host_state.numel() * 4,
                    "d2h_bytes_per_step": host_state.numel() * 4 + 9 * G + host_cnt.numel() * 8, "steps": e2e_steps},
            "gpu_launches": steps,
            "roofline": {"bound": "tensor", "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak,
                         "traffic": profiled("policy_p2_%s_g%d_k%d" % ("lid" if ctx.pool else "random", G, K)),
                         "peak_source": "measured (MEASURED_PEAKS.json bf16_tflops, burst)" if peaks else "fallback",
                         "algorithmic_flop_per_decision": flop, "decisions_per_launch": G * K,
                         "kernel": "pol::k_policy_rollout<%d>" % ctx.pool},
            "clocks": clocks, "decisions_per_sec": value, "games_per_sec": (cnt[1] / max(cnt[0], 1)) * value,
            "accuracy": accuracy, "rollout_counters": {"steps": cnt[0], "games": cnt[1], "rounds": cnt[2], "stuck": cnt[6]},
            "outputs": outputs}


def measure_train(args, ctx, games, steps, warmup):
    """BASELINE.json configs[4]: the scripts/training.py-equivalent loop -- GPU self-play rollouts of `games` episodes
    per rank against the random opponent + one A2C update with a flat NCCL gradient all-reduce per bench step.  The
    timed region runs the product's training step (SelfPlayTrainer.step: the whole batch as one CUDA graph); a few
    launch-by-launch batches before it give the rollout / update split."""
    torch = ctx.torch
    from azul_deep_reinforcement_learning_b200.train import SelfPlayTrainer
    tr = SelfPlayTrainer(games, seed=args.seed & 0x7FFFFFFF, device=ctx.local, rank=ctx.rank, world=ctx.world)
    steps_word = lambda: int(tr.runner.engine.state[6].to(torch.int64).sum())   # noqa: E731  env steps executed so far
    for _ in range(warmup):
        tr.update(tr.rollout())
    upd_ms, roll_ms, sync_ms, trans = [], [], [], 0.0
    for _ in range(3):                               # launch by launch, synchronised: where the time goes
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        batch = tr.rollout()
        torch.cuda.synchronize()
        t1 = time.perf_counter()
        st = tr.update(batch)
        torch.cuda.synchronize()
        upd_ms.append(1e3 * (time.perf_counter() - t1)); roll_ms.append(1e3 * (t1 - t0))
        sync_ms.append(1e3 * st.get("update_sync_s", 0.0)); trans = st["transitions"]
    graph = not args.no_graph
    if graph:
        tr.enable_step_graph(warmup=1)
    ctx.barrier()
    sampler = ctx.clocks()
    if ctx.rank == 0:
        sampler.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s0 = steps_word()
    ctx.barrier()
    ev0.record()
    for _ in range(steps):
        tr.step(defer_stats=True)
    ev1.record()
    ctx.barrier()
    clocks = sampler.stop() if ctx.rank == 0 else None
    last = None
    for _ in range(steps):
        last = tr.fetch_stats()                      # every batch's statistics reached the host
    outputs = None
    if args.dump_outputs:                        # the trained network and the last batch's statistics (not its host wait time)
        outputs = ({}, {**{"param." + n: p.detach() for n, p in tr.net.named_parameters()},
                        **{"stat." + k: torch.tensor(float(v), dtype=torch.float64) for k, v in last.items() if k != "update_sync_s"}})
    env_steps, n_games = steps_word() - s0, games * steps
    dev_ms = ctx.max_over_ranks(ev0.elapsed_time(ev1))
    tot = torch.tensor([float(env_steps), float(n_games)], dtype=torch.float64, device=ctx.dev)
    ctx.parallel.reduce_counters(tot)
    cfg = workload_config(args, ctx.world, games=games, players=2)
    cfg["workload"] = ("self-play A2C training: %d episodes per GPU per batch vs the random opponent (persistent fused policy "
                       "kernel rollouts), discounted returns, Agent.update loss and gradients on the tensor cores, fused Adam, flat "
                       "NCCL gradient all-reduce; %s (BASELINE.json configs[4])" % (
                           games, "one CUDA graph per batch" if graph else "launch by launch"))
    cfg.pop("env_steps_per_game_per_launch", None)
    cfg["l2"] = "n/a (multi-kernel training step; working set is re-generated every batch)"
    value = float(tot[0]) / (dev_ms * 1e-3)
    return {"value": value, "unit": UNIT, "n_gpus": ctx.world, "steps": steps, "warmup": warmup + 3, "ms_per_step": dev_ms / steps,
            "dtype": "fp16-operand tensor-core MLP (rollout and update), fp32 accumulation / u32 rules", "config": cfg,
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 8 * 18,
                    "note": "a training batch is end to end by construction: its statistics are copied to pinned host memory every batch"},
            # this library's kernels per batch: pack weights, reset, opponent loop (reset), persistent policy rollout,
            # returns, statistics, update forward/backward, update dW (plus torch fills / reductions / fused Adam / NCCL)
            "gpu_launches": 8 * steps, "clocks": clocks,
            "games_per_sec": float(tot[1]) / (dev_ms * 1e-3), "agent_decisions_per_batch": trans,
            "rollout_ms": statistics.median(roll_ms), "update_ms": statistics.median(upd_ms),
            "allreduce_and_stats_ms": statistics.median(sync_ms), "cuda_graph": graph,
            "launch_by_launch_step_ms": [round(a + b, 2) for a, b in zip(roll_ms, upd_ms)],
            "last_batch": {k: last[k] for k in ("reward", "ac_loss", "win_percent", "unfinished")} if last else None,
            "outputs": outputs}


def finish_line(args, m, extra_keys=()):
    """A measurement dict -> the contract's JSON line."""
    line = {"metric": METRIC, "value": m["value"], "unit": UNIT, "n_gpus": m["n_gpus"], "steps": m["steps"],
            "warmup": m["warmup"], "ms_per_step": m["ms_per_step"], "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": m.get("dtype", "u32"), "data": "synthetic", "config": m["config"]}
    for k, v in m.items():
        if k not in line and k != "outputs":
            line[k] = v
    return line


DUMP_BYTES = 63 * 10 ** 6           # array data; the .npy headers stay within the 64 MB of --dump-outputs


def dump_outputs(out_dir, per_game, whole):
    """--dump-outputs: one DIR/<name>.npy per tensor, integers as float64 (exact for 32-bit words and the counters),
    floating point as float32 (float64 stays float64).  ``per_game`` tensors have the game as their last axis; when
    everything does not fit DUMP_BYTES, all of them keep the same seeded sample of games, listed in game_index.npy."""
    import numpy as np
    import torch
    wide = lambda t: not t.is_floating_point() or t.dtype == torch.float64      # noqa: E731  written as float64
    fixed = sum(t.numel() * (8 if wide(t) else 4) for t in whole.values())
    per = sum(t[..., 0].numel() * (8 if wide(t) else 4) for t in per_game.values())
    n = next(iter(per_game.values())).shape[-1] if per_game else 0
    os.makedirs(out_dir, exist_ok=True)
    if fixed + n * per > DUMP_BYTES:
        keep = (DUMP_BYTES - fixed) // (per + 8)
        assert keep > 0, "--dump-outputs: the outputs without a game axis alone exceed the budget"
        idx = np.sort(np.random.default_rng(0).choice(n, keep, replace=False))
        np.save(os.path.join(out_dir, "game_index.npy"), idx.astype(np.float64))
        per_game = {k: v.index_select(-1, torch.from_numpy(idx).to(v.device)) for k, v in per_game.items()}
    for name, t in {**per_game, **whole}.items():
        t = t.detach()
        np.save(os.path.join(out_dir, name + ".npy"), (t.double() if wide(t) else t.float()).cpu().numpy())


def run_b200(args):
    ctx = Ctx(args)
    warm = max(args.warmup, 3)
    mode = args.mode
    if mode == "step":
        head = measure_step(args, ctx, args.games, args.players, args.steps, warm)
        line = finish_line(args, head)
    elif mode == "policy":
        head = measure_policy(args, ctx, args.games, args.steps, warm)
        line = finish_line(args, head)
    elif mode == "train":
        head = measure_train(args, ctx, args.games, args.steps, warm)
        line = finish_line(args, head)
    elif mode == "config3":
        ms = {"p%d" % p: measure_random(args, ctx, p, args.games, args.steps, warm, e2e=False) for p in (2, 3, 4)}
        head = ms["p%d" % args.players]
        line = finish_line(args, head)
        line["config3"] = {k: {kk: v[kk] for kk in ("value", "ms_per_step", "roofline", "clocks", "games_per_sec")} for k, v in ms.items()}
    else:
        head = measure_random(args, ctx, args.players, args.games, args.steps, warm, e2e=True)
        line = finish_line(args, head)
        if not args.no_extras:
            # the rest of SURVEY §8(d), measured in the same process right after the headline (each with its own clocks)
            brief = ("value", "unit", "ms_per_step", "steps", "e2e", "roofline", "clocks", "games_per_sec", "config", "gpu_launches")
            extra = {}
            es = max(3, min(args.steps, 20))
            m = measure_step(args, ctx, 1 << 22, 2, es, 3)
            extra["step"] = {k: m[k] for k in brief if k in m}
            extra["config3"] = {}
            for p in (2, 3, 4):
                m = measure_random(args, ctx, p, 262144, max(3, min(args.steps, 5)), 3, e2e=False)
                extra["config3"]["p%d" % p] = {k: m[k] for k in brief if k in m and k != "e2e"}
            m = measure_policy(args, ctx, 131072, es, 3)
            extra["policy"] = {k: m[k] for k in brief + ("decisions_per_sec", "accuracy", "dtype") if k in m}
            m = measure_train(args, ctx, 16384, max(3, min(args.steps, 8)), 3)
            extra["train"] = {k: m[k] for k in brief + ("agent_decisions_per_batch", "rollout_ms", "update_ms", "allreduce_and_stats_ms", "launch_by_launch_step_ms", "cuda_graph", "last_batch", "dtype") if k in m}
            line["extra"] = extra
    if ctx.rank == 0:
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, *head["outputs"])
        if ctx.world == 1 and not args.no_cpu_baseline and mode == "random":
            threads = os.cpu_count() or 1
            v, n, k, dt = cpu_rollout_rate(args, args.cpu_seconds, threads)
            line["cpu_baseline"] = {
                "value": v, "unit": UNIT, "cores": threads, "kind": "port", "cpu_model": cpu_model_name(),
                "sample": "%d of %d games x %d env steps (bounded sample: the rate does not depend on the batch size), "
                          "C oracle port on %d threads, %.1f s" % (n, args.games, k, threads, dt)}
            py = python_reference_leg(args.pyref_seconds)
            if py is not None:
                line["cpu_baseline"]["python_reference"] = py
            if "extra" in line and args.pyref_seconds > 0:
                # the same reference, on the paths of configs[3] / configs[4] (shorter legs: the rate settles within seconds)
                short = min(args.pyref_seconds, 10.0)
                line["extra"]["policy"]["cpu_python_reference"] = python_reference_leg(short, "selfplay")
                line["extra"]["train"]["cpu_python_reference"] = python_reference_leg(short, "train")
        print(json.dumps(line))
    ctx.close()


def main():
    args = parse_args()
    if args.pyref_worker is not None:
        return pyref_worker(args.pyref_worker, args.pyref_kind)
    if not args.games:
        args.games = {"policy": 131072, "train": 16384, "step": 1 << 22, "config3": 262144}.get(args.mode, 65536)
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
