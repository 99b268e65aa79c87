#!/usr/bin/env python
"""bench.py — env-steps/s of the batched CookingZoo step + feature_vector observation path.

    python bench.py [--gpus N] [--steps K] [--warmup W]            # this repo's CUDA path
    python bench.py --impl reference [--gpus N] [--steps K] ...    # CPU baseline arm (oracle port)
    python bench.py ... --dump-outputs DIR                         # also write the last timed step's outputs to DIR/*.npy

One "step" = one cz_step launch advancing every environment of this rank once (each agent acts,
rewards / termination / truncation computed, every agent's float64 feature vector written).
Workload (BASELINE.json configs[3], the configuration the metric is quoted on): 1 Mi
two-agent coop_test environments sharded over 8 GPUs = 131072 environments per GPU (weak
scaling: per-GPU work is fixed), per-environment recipe pairs drawn from the 8-recipe book,
uniform random actions resident in HBM, max_steps 400 with auto-reset from the layout pool.
The per-step working set (observations 583 MB + state 19 MB per GPU) is larger than the
126 MB L2, so no explicit L2 flush is needed between steps.
"""
import argparse
import json
import multiprocessing as mp
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

ENVS_PER_GPU = 131072
NUM_AGENTS = 2
MAX_STEPS = 400
LEVEL, META = "coop_test", "example"
BOOK = ["TomatoSalad", "TomatoLettuceSalad", "CarrotBanana", "MashedCarrotBanana", "CucumberOnion",
        "AppleWatermelon", "TomatoLettuceOnionSalad", "no_recipe"]
METRIC = "env-steps/sec (batched step+feature_vector obs)"
UNIT = "env-steps/s"
BACKGROUND_DYN_BLOCKS = 0     # pipelined block: dynamics grid of step k+1 (0 = full grid; with the whole-row TMA writer a capped grid no longer pays)
FALLBACK_HBM_GBS = 6650.0     # /opt/skills/guides/B200_PROFILING.md, used only if MEASURED_PEAKS.json is absent


def bind_to_gpu_numa_node(local):
    """Pin this rank to the CPUs of its GPU's NUMA node, so that the pinned host buffers of the e2e leg (first touch)
    and the copy-engine traffic stay on the socket the GPU hangs off.  Best effort: returns the node or None."""
    try:
        import torch
        pr = torch.cuda.get_device_properties(local)
        path = f"/sys/bus/pci/devices/{pr.pci_domain_id:04x}:{pr.pci_bus_id:02x}:{pr.pci_device_id:02x}.0/numa_node"
        node = int(open(path).read().strip())
        if node < 0:
            return None
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            return node
    except Exception:
        pass
    return None


def workload_config(n_gpus, envs_per_gpu):
    return {"workload": f"cfg4 shard: {envs_per_gpu} envs/GPU x {n_gpus} GPU, coop_test/example, 2 agents, "
                        f"per-env recipe pairs from the 8-recipe book, scheme3 uniform random actions, "
                        f"max_steps {MAX_STEPS}, auto-reset from the exact 400-layout distribution of the level parser, "
                        f"feature_vector f64 obs",
            "envs_per_gpu": envs_per_gpu, "num_agents": NUM_AGENTS, "obs_len": 278,
            "l2": "per-step working set (>600 MB) exceeds the 126 MB L2; no flush needed",
            "parallelism": f"env-sharded x{n_gpus}, no per-step collective"}


# ------------------------------------------------------------------------------------------
# clocks: sampled with NVML from a thread while the timed region runs
# ------------------------------------------------------------------------------------------
class ClockSampler:
    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown",
               0x4: "sw_power_cap", 0x80: "hw_power_brake", 0x2: "applications_clocks_setting"}

    def __init__(self, index):
        self.samples, self.stop_flag, self.thread, self.h = [], False, None, None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.h = None

    def _run(self):
        nv = self.nv
        while not self.stop_flag:
            try:
                mhz = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
                try:
                    rs = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    rs = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                self.samples.append((time.perf_counter(), mhz, rs))
            except Exception:
                pass
            time.sleep(0.01)

    def start(self):
        if self.h is not None:
            self.thread = threading.Thread(target=self._run, daemon=True)
            self.thread.start()

    def stop(self, t0, t1):
        if self.h is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvml unavailable"]}
        self.stop_flag = True
        self.thread.join()
        inside = [s for s in self.samples if t0 <= s[0] <= t1] or self.samples[-3:]
        reasons = set()
        for _, _, rs in inside:
            for bit, name in self.REASONS.items():
                if rs & bit:
                    reasons.add(name)
        return {"sm_mhz": float(np.median([s[1] for s in inside])) if inside else None,
                "sm_max_mhz": float(self.max_mhz), "samples": len(inside), "reasons": sorted(reasons)}


# ------------------------------------------------------------------------------------------
# CPU arm: the oracle port on the host cores (the reference itself is Python and cannot travel
# to the GPU box; oracle/cz_oracle.py is its pinned restatement, same language, same structure)
# ------------------------------------------------------------------------------------------
def _cpu_worker(args):
    wid, n_steps, warm, seed = args
    import random
    from oracle.cz_oracle import OracleEnv
    from cooking_zoo_b200.layout import sample_layout
    from cooking_zoo_b200.levels import load_level_object, load_meta
    rng = np.random.default_rng(seed * 1000 + wid)
    lay_rng = random.Random(seed * 1000 + wid)
    level, meta = load_level_object(LEVEL), load_meta(META)

    def fresh():
        rec = [BOOK[int(rng.integers(8))], BOOK[int(rng.integers(8))]]
        return OracleEnv(sample_layout(level, meta, NUM_AGENTS, lay_rng), rec, MAX_STEPS, end_condition_all_dishes=True)

    env = fresh()
    acts = rng.integers(0, 5, size=(n_steps + warm, NUM_AGENTS))
    t0 = None
    for s in range(n_steps + warm):
        if s == warm:
            t0 = time.perf_counter()
        _, term, trunc, _ = env.step(acts[s])
        env.observe(0)
        env.observe(1)
        if any(term) or any(trunc):
            env = fresh()
    return time.perf_counter() - t0


def cpu_port_throughput(steps_per_worker, warm, procs=None):
    procs = procs or os.cpu_count() or 1
    ctx = mp.get_context("spawn")
    with ctx.Pool(procs) as pool:
        t0 = time.perf_counter()
        times = pool.map(_cpu_worker, [(w, steps_per_worker, warm, 7) for w in range(procs)])
        wall = time.perf_counter() - t0
    total = steps_per_worker * procs
    return total / max(times), procs, wall


def _ref_worker(args):
    """One process of the reference arm: the UNMODIFIED reference environment (oracle/_ref or /root/reference behind the
    import stubs of oracle/refshim), driven below its PettingZoo wrapper exactly as SURVEY.md §8(c) prescribes:
    accumulated_step(actions) + observe(agent) for every agent, reset() when the episode ends."""
    wid, n_steps, warm, seed = args
    import random
    from oracle.ref_loader import load_reference
    ce = load_reference()
    random.seed(seed * 1000 + wid)
    np.random.seed(seed * 1000 + wid)
    rng = np.random.default_rng(seed * 1000 + wid)
    rec = [BOOK[int(rng.integers(8))], BOOK[int(rng.integers(8))]]
    env = ce.CookingEnvironment(level=LEVEL, meta_file=META, num_agents=NUM_AGENTS, max_steps=MAX_STEPS, recipes=rec,
                                obs_spaces=["feature_vector"] * NUM_AGENTS, end_condition_all_dishes=True,
                                action_scheme="scheme3")
    env.reset()
    agents = list(env.possible_agents)
    acts = rng.integers(0, 5, size=(n_steps + warm, NUM_AGENTS)).tolist()
    t0 = None
    for s in range(n_steps + warm):
        if s == warm:
            t0 = time.perf_counter()
        env.accumulated_step(acts[s])
        for a in agents:
            env.observe(a)
        if any(env.terminations.values()) or any(env.truncations.values()):
            env.reset()
    return time.perf_counter() - t0


def reference_available():
    try:
        from oracle.ref_loader import reference_available as ok
        return ok()
    except Exception:
        return False


def cpu_reference_throughput(steps_per_worker, warm, procs=None):
    procs = procs or os.cpu_count() or 1
    ctx = mp.get_context("spawn")
    with ctx.Pool(procs) as pool:
        t0 = time.perf_counter()
        times = pool.map(_ref_worker, [(w, steps_per_worker, warm, 7) for w in range(procs)])
        wall = time.perf_counter() - t0
    return steps_per_worker * procs / max(times), procs, wall


def cpu_port_c_throughput(n_envs=4096, steps=60, warm=5):
    """The compiled restatement (oracle/cz_oracle.c) on all host threads: an honest compiled-CPU data point
    beside the Python-port baseline (the reference itself is Python)."""
    import random
    from oracle.cz_oracle_c import CBatch
    from cooking_zoo_b200.layout import sample_layout
    from cooking_zoo_b200.levels import load_level_object, load_meta
    rng = np.random.default_rng(5)
    lay_rng = random.Random(5)
    level, meta = load_level_object(LEVEL), load_meta(META)
    pool = [sample_layout(level, meta, NUM_AGENTS, lay_rng) for _ in range(64)]
    threads = os.cpu_count() or 1
    batch = CBatch([pool[i % 64] for i in range(n_envs)],
                   [[BOOK[int(rng.integers(8))], BOOK[int(rng.integers(8))]] for _ in range(n_envs)], 10 ** 6,
                   threads=threads, end_condition_all_dishes=True)
    acts = rng.integers(0, 5, size=(steps + warm, n_envs, NUM_AGENTS)).astype(np.uint8)
    for s in range(warm):
        batch.step(acts[s])
    t0 = time.perf_counter()
    for s in range(warm, warm + steps):
        batch.step(acts[s])
    dt = time.perf_counter() - t0
    return n_envs * steps / dt, threads


def run_reference_arm(args):
    """bench.py --impl reference: the reference's own CPU implementation of the path on every host core.  The reference
    is pure Python; `python -m oracle.make_ref` (run by __graft_entry__.build()) copies it verbatim into the git-ignored
    oracle/_ref/, which travels to the box.  Only when that copy is missing does the arm fall back to the oracle port
    (kind "port")."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    # each "step" = every host core advances its own environment once
    timed, warm = args.steps, args.warmup
    extra = {}
    if reference_available():
        kind = "reference"
        value, procs, wall = cpu_reference_throughput(timed, warm)
        from oracle.ref_loader import REFERENCE_ROOT
        what = (f"the unmodified reference (cooking_zoo.environment.cooking_env.CookingEnvironment from {REFERENCE_ROOT}, "
                f"behind the import stubs of oracle/refshim): accumulated_step + observe() for both agents, reset() on episode end")
        try:        # the oracle port beside it (informational: same loop, the restatement instead of the reference)
            pv, _, _ = cpu_port_throughput(timed, warm)
            extra["oracle_port"] = {"value": pv, "unit": UNIT, "cores": procs, "kind": "port"}
        except Exception as ex:
            extra["oracle_port"] = {"unavailable": str(ex)[:120]}
    else:
        kind = "port"
        value, procs, wall = cpu_port_throughput(timed, warm)
        what = "the oracle port (oracle/cz_oracle.py): oracle/_ref is missing, run `python -m oracle.make_ref`"
    ms = 1000.0 * procs / value
    sample = (f"{procs} processes x ({warm} warm-up + {timed} timed) env-steps of {what}; one two-agent coop_test "
              f"environment per process, recipe pair drawn from the 8-recipe book, uniform random scheme3 actions")
    cfg = workload_config(args.gpus, ENVS_PER_GPU)
    cfg["reference_arm"] = (f"same environment configuration, stepped as {procs} independent single-environment processes "
                            f"(a multiprocessing vector env over the host cores), not as one {ENVS_PER_GPU}-environment batch")
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": cfg,
            "cpu_baseline": dict({"value": value, "unit": UNIT, "cores": procs, "kind": kind, "sample": sample}, **extra),
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    emit(line)


# ------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------
def run_gpu_arm(args):
    import torch
    import torch.distributed as dist
    from cooking_zoo_b200 import BatchedCookingEnv
    from cooking_zoo_b200 import _native

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local}"))
    torch.cuda.set_device(local)
    numa_node = bind_to_gpu_numa_node(local) if world > 1 else None
    dev = torch.device(f"cuda:{local}")
    N, A = args.envs, NUM_AGENTS

    L = None
    g = torch.Generator(device="cpu").manual_seed(1234 + rank)
    recipe_ids = torch.randint(0, len(BOOK), (N, 2), generator=g, dtype=torch.uint8)
    ring = 16
    actions = torch.randint(0, 5, (ring, N, A), generator=g, dtype=torch.uint8).to(dev)

    def sync_all():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize(dev)

    def timed_run(pipelined, sample_clocks, obs_dtype=torch.float64, background=BACKGROUND_DYN_BLOCKS, force_eager=False):
        """W warm-up + K timed steps of one mode; returns (env, ms_total max over ranks, launches, clocks, how).

        The K timed steps are enqueued as ONE CUDA graph when K <= 512 (captured after the eager warm-up, replayed once
        untimed, then timed): the driver's short runs (K = 20) otherwise measure the host's launch jitter, not the GPU.
        Every step is a full cz_step / cz_step_pipelined with its own resident action tensor; nothing is skipped."""
        env = BatchedCookingEnv(N, LEVEL, META, A, MAX_STEPS, BOOK[1:3], end_condition_all_dishes=True, action_scheme="scheme3",
                                device=str(dev), recipe_pool=BOOK, layout_pool_size="auto", layout_seed=0,
                                auto_reset=True, seed=2026, env_offset=rank * N, pipelined=pipelined, obs_dtype=obs_dtype,
                                background_dynamics=background if pipelined else 0)
        env.reset(recipe_ids=recipe_ids)
        for s in range(args.warmup):
            env.step(actions[s % ring])
        env.wait()
        sync_all()
        K = args.steps
        graph, how = None, "eager launches"
        # steps per graph: K itself up to 512, else the largest divisor of K that is at most 256 (K = 2000 -> 10 replays of 200)
        G = K if K <= 512 else max((g for g in range(1, 257) if K % g == 0), default=1)
        if not args.no_graph and not force_eager and G >= 10 and (not pipelined or G % 2 == 0):
            try:
                if pipelined:   # no event of the eager warm-up may be waited on inside the capture
                    _native.check(env.lib.cz_pipeline_reset(env._handle, env.lib.cz_pipeline_current(env._handle)))
                side = torch.cuda.Stream(dev)
                side.wait_stream(torch.cuda.current_stream(dev))
                graph = torch.cuda.CUDAGraph()
                l0 = env.lib.cz_launch_count()
                with torch.cuda.stream(side):
                    with torch.cuda.graph(graph, stream=side, capture_error_mode="thread_local"):
                        for s in range(G):
                            env.step(actions[s % ring])
                        env.wait()
                captured = (env.lib.cz_launch_count() - l0) * (K // G)
                torch.cuda.current_stream(dev).wait_stream(side)
                graph.replay()          # untimed: G more warm-up steps, uploads the graph
                how = (f"one CUDA graph of the {K} steps ({captured} kernel nodes)" if G == K else
                       f"{K // G} replays of one CUDA graph of {G} steps ({captured} kernel launches)")
            except Exception as ex:     # capture not possible on this box: time eager launches
                sys.stderr.write(f"timed_run: graph capture failed ({ex!r}); timing eager launches\n")
                graph = None
                env.close()
                return timed_run_eager(pipelined, sample_clocks, obs_dtype)
        sync_all()
        sampler = ClockSampler(local) if sample_clocks else None
        if sampler:
            sampler.start()
        launches0 = env.lib.cz_launch_count()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        sync_all()
        t_host0 = time.perf_counter()
        # keep the stream busy for ~0.1 ms while the host enqueues the opening event and the first launch: the timed region then
        # starts on the device with its first kernel already queued, instead of with the host's launch latency
        if not os.environ.get("CZ_BENCH_NO_PRIME"):
            torch.cuda._sleep(200000)
        ev0.record()
        if graph is not None:
            for _ in range(K // G):
                graph.replay()
        else:
            for s in range(K):
                env.step(actions[s % ring])
            env.wait()      # pipelined mode: order the internal streams before the closing event (no-op otherwise)
        ev1.record()
        torch.cuda.synchronize(dev)
        t_host1 = time.perf_counter()
        if graph is not None and pipelined:
            # the library's events were last recorded inside the capture: forget them before any eager call waits on one
            _native.check(env.lib.cz_pipeline_reset(env._handle, env.lib.cz_pipeline_current(env._handle)))
        launches = captured if graph is not None else env.lib.cz_launch_count() - launches0
        clocks = sampler.stop(t_host0, t_host1) if sampler else None
        if not os.environ.get("CZ_BENCH_NO_PRIME"):
            how += "; a ~0.1 ms spin kernel in front of the opening event keeps the host's launch latency out of the device-timed region"
        t = torch.tensor([ev0.elapsed_time(ev1)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.barrier()
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        env._bench_graph = graph        # keep the graph (and its captured pointers) alive as long as the environment
        # the steps this environment took (warm-up, the graph's untimed replay, timed) and the steps per graph (0: eager
        # launches): with a graph, step s of each replay takes actions[s % ring], so the last step's outputs depend on it
        env._bench_schedule = (args.warmup, G if graph is not None else 0, K, G if graph is not None else 0)
        return env, float(t.item()), launches, clocks, how

    def timed_run_eager(pipelined, sample_clocks, obs_dtype):
        args.no_graph = True
        return timed_run(pipelined, sample_clocks, obs_dtype)

    # the other step mode first (reported as a block of the line), then the headline mode with the clocks sampled:
    # --mode sync (default): the in-place step is the headline, the two-stream pipelined mode the block, and vice versa
    head_pipe = args.mode == "pipelined"
    env_s, ms_other, launches_other, _, how_other = timed_run(not head_pipe, False)
    other_value = world * N * args.steps / (ms_other / 1e3)
    L = env_s.obs_len
    env_s.wait()
    env_s.close()
    del env_s
    torch.cuda.empty_cache()
    # the pipelined step with a capped background dynamics grid needs eager launches with the whole-row writer (inside a graph
    # the capped grid loses, profiles/r02_notes.md §17): reported as a second figure of the pipelined block
    try:
        if args.no_bg:
            raise RuntimeError("skipped (--no-bg)")
        env_b, ms_bg, _, _, how_bg = timed_run(True, False, background=3, force_eager=True)
        env_b.wait()
        env_b.close()
        del env_b
        torch.cuda.empty_cache()
        bg_block = {"value": world * N * args.steps / (ms_bg / 1e3), "ms_per_step": ms_bg / args.steps, "timed_region": how_bg,
                    "how": "cz_pipeline_config(2 state matrices, 3 dynamics blocks per SM), eager launches"}
    except Exception as ex:
        bg_block = {"error": f"{type(ex).__name__}: {str(ex)[:160]}"}
    env, ms_total_max, launches, clocks, how_timed = timed_run(head_pipe, True)
    if args.dump_outputs and rank == 0:
        dump_outputs(env, args.dump_outputs)       # before the e2e leg below steps the same state further
    lib = env.lib
    ms_per_step = ms_total_max / args.steps
    value = world * N * args.steps / (ms_total_max / 1e3)

    # optional episode statistics, reduced once with NCCL (not on the per-step path)
    info = env.info()
    stats = torch.stack([(env.state[env.tables.num_dyn_slots + A + 5].to(torch.float64)).sum(),
                         info["recipe_done"].to(torch.float64).sum(), env.reward.sum()])
    if world > 1:
        dist.all_reduce(stats, op=dist.ReduceOp.SUM)

    # ---- e2e: the reference-facing call with HOST buffers (cz_step_host), copies inside the timed region
    e2e_steps = max(3, min(args.steps, args.e2e_steps))
    h_act = torch.randint(0, 5, (N, A), generator=g, dtype=torch.uint8).pin_memory()
    h_obs = torch.empty((N, A, L), dtype=torch.float64).pin_memory()
    h_rew = torch.empty((N, A), dtype=torch.float64).pin_memory()
    h_term = torch.empty((N, A), dtype=torch.uint8).pin_memory()
    h_trunc = torch.empty((N, A), dtype=torch.uint8).pin_memory()
    stream = torch.cuda.current_stream(dev).cuda_stream

    env.wait()
    torch.cuda.synchronize(dev)

    def host_step():
        _native.check(lib.cz_step_host(env._handle, env.state.data_ptr(), h_act.data_ptr(), h_obs.data_ptr(),
                                       h_rew.data_ptr(), h_term.data_ptr(), h_trunc.data_ptr(), N,
                                       _native.STEP_AUTO_RESET, 2026, rank * N, stream))
    for _ in range(3):
        host_step()
    sync_all()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(e2e_steps):
        host_step()
    e1.record()
    torch.cuda.synchronize(dev)
    te = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_value = world * N * e2e_steps / (float(te.item()) / 1e3)
    h2d = N * A
    d2h = N * A * L * 8 + N * A * 8 + 2 * N * A

    # ---- BASELINE config 3 (4096 two-agent envs on one GPU): latency-bound; per launch and K steps per launch
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        peak, peak_src = float(json.load(open(peaks_path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    else:
        peak, peak_src = FALLBACK_HBM_GBS, "fallback (B200_PROFILING.md)"

    def rate(fn, units, reps, warm=5, fin=None):
        for _ in range(warm):
            fn()
        if fin:
            fin()
        torch.cuda.synchronize(dev)
        a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a0.record()
        for _ in range(reps):
            fn()
        if fin:
            fin()       # pipelined groups: order the internal streams before the closing event
        a1.record()
        torch.cuda.synchronize(dev)
        return units * reps / (a0.elapsed_time(a1) / 1e3)

    only = set(filter(None, os.environ.get("CZ_BENCH_ONLY", "").split(",")))      # e.g. CZ_BENCH_ONLY=cfg5 while tuning

    def want(name):
        return rank == 0 and world == 1 and not args.no_cfg3 and (not only or name in only)

    cfg3 = None
    if want("cfg3"):
        try:
            n3, K3 = 4096, 64
            env3 = BatchedCookingEnv(n3, LEVEL, META, A, MAX_STEPS, BOOK[1:3], end_condition_all_dishes=True, action_scheme="scheme3",
                                     device=str(dev), layout_pool_size="auto", layout_seed=0, auto_reset=True, seed=7)
            env3.reset()
            act3 = torch.randint(0, 5, (K3, n3, A), generator=g, dtype=torch.uint8).to(dev)
            cnt = [0]

            def one_step():
                env3.step(act3[cnt[0] % K3])
                cnt[0] += 1
            per_launch = rate(one_step, n3, 2000, 20)
            # K steps in ONE launch of the warp-per-environment kernel (cz_step's k_steps): actions of the K steps resident,
            # or drawn inside the kernel from the counter stream of cz_random_actions
            k_res = rate(lambda: env3.step_k(K3, actions=act3), n3 * K3, 60)
            k_dev = rate(lambda: env3.step_k(K3, action_step=cnt[0]), n3 * K3, 60)
            # the same per-step launches captured in a CUDA graph (what round 1 reported as its K-step figure)
            graph = torch.cuda.CUDAGraph()
            side = torch.cuda.Stream(dev)
            side.wait_stream(torch.cuda.current_stream(dev))
            with torch.cuda.stream(side):
                with torch.cuda.graph(graph, stream=side, capture_error_mode="thread_local"):
                    for s in range(16):
                        env3.step(act3[s])
            torch.cuda.current_stream(dev).wait_stream(side)
            graphed = rate(graph.replay, n3 * 16, 200)
            b3 = A * env3.obs_len * 8 + A * 8 + 2 * A + A + 2 * env3.tables.rows * 4
            cfg3 = {"workload": "cfg3: 4096 two-agent coop_test envs, 1 GPU, random actions, feature_vector f64 obs, auto-reset",
                    "per_launch_env_steps_per_s": per_launch,
                    "cuda_graph_env_steps_per_s": graphed,
                    "k_steps_per_launch": {"K": K3, "env_steps_per_s": k_res,
                                           "how": f"cz_step(k_steps={K3}): one launch of cz_warp_kernel (one warp per environment, "
                                                  f"state in registers across the K steps, rows written every step), actions "
                                                  f"[K][n][A] resident",
                                           "device_actions_env_steps_per_s": k_dev,
                                           "device_actions_how": "the same launch with CZ_STEP_DEVICE_ACTIONS: actions drawn inside "
                                                                 "the kernel from the counter stream of cz_random_actions"},
                    "bytes_per_env_step": b3,
                    "roofline": {"bound": "latency (19 MB of rows per step stay in the 126 MB L2)", "unit": "GB/s",
                                 "achieved": k_res * b3 / 1e9, "peak": peak, "frac": k_res * b3 / 1e9 / peak},
                    "note": "a step writes 19 MB: bounded by the per-step instruction chain, not by HBM"}
            env3.close()
        except Exception as ex:      # a side measurement must never cost the headline line
            cfg3 = {"error": f"{type(ex).__name__}: {str(ex)[:200]}"}

    # ---- BASELINE config 5: 1-4 agents per environment, heuristic cooks on the device, despawn / respawn on
    cfg5 = None
    if want("cfg5"):
        try:
            from cooking_zoo_b200 import MixedAgentCookingEnv
            n5 = args.cfg5_envs
            counts = (np.arange(n5) % 4) + 1
            lv5 = os.path.join(ROOT, "tests", "golden", "levels", "open4.json")
            mt5 = os.path.join(ROOT, "tests", "golden", "levels", "meta4.json")
            r5 = ["TomatoLettuceSalad", "CarrotBanana", "TomatoSalad", "AppleWatermelon"]
            out5, b5 = {}, 0.0
            for mode in ("in_place", "pipelined"):
                try:
                    mix = MixedAgentCookingEnv(counts, lv5, mt5, MAX_STEPS, r5, device=str(dev), end_condition_all_dishes=True,
                                               action_scheme="scheme3", layout_pool_size=256, auto_reset=True, seed=5,
                                               agent_respawn_rate=0.2, agent_despawn_rate=0.05, grace_period=3,
                                               pipelined=(mode == "pipelined"))
                    mix.reset()
                    b5 = sum(len(mix.index[a]) * (a * grp.obs_len * 8 + a * 11 + 2 * grp.tables.rows * 4)
                             for a, grp in mix.groups.items()) / n5
                    for _ in range(5):
                        mix.cook_step()
                    mix.wait()
                    torch.cuda.synchronize(dev)
                    # 10 closed-loop steps (per group: cz_policy_act + step on the group's stream) as one CUDA graph: the
                    # eager loop is bound by the host's per-group launch work, not by the GPU
                    graph5 = torch.cuda.CUDAGraph()
                    side = torch.cuda.Stream(dev)
                    side.wait_stream(torch.cuda.current_stream(dev))
                    if mode == "pipelined":
                        for grp in mix.groups.values():
                            _native.check(grp.lib.cz_pipeline_reset(grp._handle, grp.lib.cz_pipeline_current(grp._handle)))
                    with torch.cuda.stream(side):
                        with torch.cuda.graph(graph5, stream=side, capture_error_mode="thread_local"):
                            mix.cook_steps(10)      # one fork / join of the four group streams around the 10 steps
                            mix.wait()
                    torch.cuda.current_stream(dev).wait_stream(side)
                    out5[mode] = rate(graph5.replay, n5 * 10, 20, 3)
                    out5[mode + "_eager"] = None
                    if mode == "pipelined":
                        for grp in mix.groups.values():
                            _native.check(grp.lib.cz_pipeline_reset(grp._handle, grp.lib.cz_pipeline_current(grp._handle)))
                    out5[mode + "_eager"] = rate(mix.cook_step, n5, 100, 10, fin=mix.wait)
                    mix.close()
                except Exception as ex:      # one mode failing must not cost the other
                    out5[mode] = out5.get(mode)
                    out5[mode + "_error"] = f"{type(ex).__name__}: {str(ex)[:160]}"
            cfg5 = {"workload": f"cfg5: {n5} envs on the open 4-agent kitchen, agent count 1-4 per env (one BatchedCookingEnv group per "
                                f"count, own CUDA stream each), every action from the device cook (cz_policy_act), despawn 0.05 / "
                                f"respawn 0.2 / grace 3, per-group recipes, auto-reset",
                    "closed_loop_env_steps_per_s": out5.get("in_place"), "closed_loop_pipelined_env_steps_per_s": out5.get("pipelined"),
                    "errors": {k: v for k, v in out5.items() if k.endswith("_error")},
                    "how": "10 closed-loop steps of every group captured as one CUDA graph (MixedAgentCookingEnv.cook_steps(10): four "
                           "independent stream branches, 2-3 kernels per group and step; the groups are not re-joined between steps)",
                    "size_note": "four groups share the GPU, so the rate grows with the population (profiles/r02_notes.md §5, §7, §15)",
                    "eager_env_steps_per_s": {"in_place": out5.get("in_place_eager"), "pipelined": out5.get("pipelined_eager"),
                                              "note": "host-bound: ~8 library calls and 8 stream joins per population step"},
                    "bytes_per_env_step": b5,
                    "roofline": {"bound": "hbm", "unit": "GB/s", "achieved": (out5.get("in_place") or 0) * b5 / 1e9, "peak": peak,
                                 "frac": (out5.get("in_place") or 0) * b5 / 1e9 / peak,
                                 "mode": "in place (like the headline)",
                                 "pipelined_frac": (out5.get("pipelined") or 0) * b5 / 1e9 / peak}}
        except Exception as ex:
            cfg5 = {"error": f"{type(ex).__name__}: {str(ex)[:200]}"}

    # ---- generic kernels (tables outside the specialised class; forced here with CZ_GENERIC=1 on the headline workload)
    generic = None
    if want("generic"):
        try:
            generic = {"workload": "the headline workload with the specialised classes switched off, in-place step"}
            for key, val, what in (("all_generic", "1", "cz_env_kernel<.,.,0> (tables in global memory) + cz_obs_any_kernel"),
                                   ("any_plan_writer", "2", "specialised dynamics kernel + cz_obs_any_kernel (what a custom meta "
                                                            "file outside the packed observation plans gets)")):
                os.environ["CZ_GENERIC"] = val
                envg = BatchedCookingEnv(N, LEVEL, META, A, MAX_STEPS, BOOK[1:3], end_condition_all_dishes=True,
                                         action_scheme="scheme3", device=str(dev), recipe_pool=BOOK, layout_pool_size="auto",
                                         layout_seed=0, auto_reset=True, seed=2026)
                del os.environ["CZ_GENERIC"]
                envg.reset(recipe_ids=recipe_ids)
                cg = [0]

                def gen_step():
                    envg.step(actions[cg[0] % ring])
                    cg[0] += 1
                vg = rate(gen_step, N, 100, 10)
                bg = A * envg.obs_len * 8 + A * 8 + 2 * A + A + 2 * envg.tables.rows * 4
                generic[key] = {"kernels": what, "env_steps_per_s": vg,
                                "roofline": {"bound": "hbm", "unit": "GB/s", "achieved": vg * bg / 1e9, "peak": peak,
                                             "frac": vg * bg / 1e9 / peak}}
                envg.close()
        except Exception as ex:
            os.environ.pop("CZ_GENERIC", None)
            generic = {"error": f"{type(ex).__name__}: {str(ex)[:200]}"}

    # ---- closed loop with the device policy (SURVEY §8 f3): CookingAgent decisions + step, no host in between
    cook = None
    if want("cook"):
        try:
            env.wait()
            torch.cuda.synchronize(dev)
            envc = BatchedCookingEnv(N, LEVEL, META, A, MAX_STEPS, BOOK[1:3], end_condition_all_dishes=True,
                                     action_scheme="scheme3", device=str(dev), recipe_pool=BOOK, layout_pool_size="auto",
                                     layout_seed=0, auto_reset=True, seed=2026)
            envc.reset(recipe_ids=recipe_ids)
            for _ in range(5):
                envc.step(envc.heuristic_actions()[0])
            torch.cuda.synchronize(dev)
            kc = 200
            c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            c0.record()
            for _ in range(kc):
                envc.step(envc.heuristic_actions()[0])
            c1.record()
            torch.cuda.synchronize(dev)
            loop_ms = c0.elapsed_time(c1) / kc
            c0.record()
            for _ in range(kc):
                envc.heuristic_actions()
            c1.record()
            torch.cuda.synchronize(dev)
            pol_ms = c0.elapsed_time(c1) / kc
            envc.close()
            envc = BatchedCookingEnv(N, LEVEL, META, A, MAX_STEPS, BOOK[1:3], end_condition_all_dishes=True,
                                     action_scheme="scheme3", device=str(dev), recipe_pool=BOOK, layout_pool_size="auto",
                                     layout_seed=0, auto_reset=True, seed=2026, pipelined=True)
            envc.reset(recipe_ids=recipe_ids)
            for _ in range(5):
                envc.step(envc.heuristic_actions()[0])
            envc.wait()
            torch.cuda.synchronize(dev)
            c0.record()
            for _ in range(kc):
                envc.step(envc.heuristic_actions()[0])
            envc.wait()
            c1.record()
            torch.cuda.synchronize(dev)
            loop_p_ms = c0.elapsed_time(c1) / kc
            # the same pipelined closed loop as one CUDA graph of 20 steps (what the headline's timed region is): without
            # the host's launch gaps between the three dependent kernels of a step
            graphed_p = graphed_s = None
            for pipe in (True, False):
                try:
                    envc.close()
                    envc = BatchedCookingEnv(N, LEVEL, META, A, MAX_STEPS, BOOK[1:3], end_condition_all_dishes=True,
                                             action_scheme="scheme3", device=str(dev), recipe_pool=BOOK, layout_pool_size="auto",
                                             layout_seed=0, auto_reset=True, seed=2026, pipelined=pipe)
                    envc.reset(recipe_ids=recipe_ids)
                    for _ in range(25):
                        envc.step(envc.heuristic_actions()[0])
                    envc.wait()
                    torch.cuda.synchronize(dev)
                    gc_ = torch.cuda.CUDAGraph()
                    side_c = torch.cuda.Stream(dev)
                    side_c.wait_stream(torch.cuda.current_stream(dev))
                    if pipe:
                        _native.check(lib.cz_pipeline_reset(envc._handle, lib.cz_pipeline_current(envc._handle)))
                    with torch.cuda.stream(side_c):
                        with torch.cuda.graph(gc_, stream=side_c, capture_error_mode="thread_local"):
                            for _ in range(20):
                                envc.step(envc.heuristic_actions()[0])
                            envc.wait()
                    torch.cuda.current_stream(dev).wait_stream(side_c)
                    r_ = rate(gc_.replay, N * 20, 10, 3)
                    if pipe:
                        graphed_p = r_
                        _native.check(lib.cz_pipeline_reset(envc._handle, lib.cz_pipeline_current(envc._handle)))
                    else:
                        graphed_s = r_
                except Exception as ex:
                    if pipe:
                        graphed_p = f"{type(ex).__name__}: {str(ex)[:120]}"
                    else:
                        graphed_s = f"{type(ex).__name__}: {str(ex)[:120]}"
            cook = {"workload": f"{N} two-agent envs, every action from cz_policy_act (the scripted cook)",
                    "closed_loop_env_steps_per_s": N / (loop_ms / 1e3),
                    "closed_loop_pipelined_env_steps_per_s": N / (loop_p_ms / 1e3),
                    "closed_loop_graph_env_steps_per_s": {"in_place": graphed_s, "pipelined": graphed_p,
                                                          "how": "20 closed-loop steps (cz_policy_act + step) as one CUDA graph; "
                                                                 "the two figures above are eager launches"},
                    "policy_ms_per_launch": pol_ms,
                    "policy_decisions_per_s": N * A / (pol_ms / 1e3),
                    "recipes_done_now": float(envc.info()["recipe_done"].sum())}
            envc.close()
        except Exception as ex:      # a side measurement must never cost the headline line
            cook = {"error": f"{type(ex).__name__}: {str(ex)[:200]}"}

    # ---- float32 observation mode (SURVEY §8d: reported separately; rows = the f64 rows rounded element-wise)
    f32 = None
    if want("f32"):
        try:
            env.wait()
            torch.cuda.synchronize(dev)
            envf, ms_f, _, _, _ = timed_run(True, False, torch.float32)
            envf.close()
            envf, ms_fs, _, _, _ = timed_run(False, False, torch.float32)
            h_obs32 = torch.empty((N, A, L), dtype=torch.float32).pin_memory()

            def host_step32():
                _native.check(lib.cz_step_host(envf._handle, envf.state.data_ptr(), h_act.data_ptr(), h_obs32.data_ptr(),
                                               h_rew.data_ptr(), h_term.data_ptr(), h_trunc.data_ptr(), N,
                                               _native.STEP_AUTO_RESET | _native.STEP_OBS_F32, 2026, rank * N, stream))
            for _ in range(3):
                host_step32()
            torch.cuda.synchronize(dev)
            e0.record()
            for _ in range(e2e_steps):
                host_step32()
            e1.record()
            torch.cuda.synchronize(dev)
            b32 = A * L * 4 + A * 8 + 2 * A + A + 2 * envf.tables.rows * 4
            f32 = {"dtype": "f32 observations (f64 rewards)", "bytes_per_env_step": b32,
                   "pipelined_env_steps_per_s": N * args.steps / (ms_f / 1e3),
                   "pipelined_gbs": N * b32 / (ms_f / args.steps / 1e3) / 1e9,
                   "in_place_env_steps_per_s": N * args.steps / (ms_fs / 1e3),
                   "e2e_env_steps_per_s": N * e2e_steps / (e0.elapsed_time(e1) / 1e3),
                   "d2h_bytes_per_step": N * A * L * 4 + N * A * 8 + 2 * N * A}
            envf.close()
        except Exception as ex:      # a side measurement must never cost the headline line
            f32 = {"error": f"{type(ex).__name__}: {str(ex)[:200]}"}

    if rank == 0:
        state_bytes = env.tables.rows * 4
        bytes_per_env_step = A * L * 8 + A * 8 + 2 * A + A + 2 * state_bytes
        achieved = N * bytes_per_env_step / (ms_per_step / 1e3) / 1e9
        traffic = None
        tp = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(tp):
            traffic = json.load(open(tp)).get("dram_bytes_per_launch")
        cpu = None
        if not args.no_cpu:
            port = None
            try:
                v, procs, wall = cpu_port_throughput(args.cpu_steps, 200)
                port = {"value": v, "unit": UNIT, "cores": procs, "kind": "port",
                        "sample": f"{procs} processes x {args.cpu_steps} env-steps of oracle/cz_oracle.py (Python restatement "
                                  f"of the Python reference), same level/recipes/action distribution, {wall:.1f} s wall"}
            except Exception as ex:     # e.g. no fork / spawn on the box
                port = {"unavailable": f"{type(ex).__name__}: {str(ex)[:120]}"}
            if reference_available():
                try:
                    v, procs, wall = cpu_reference_throughput(args.cpu_steps, 200)
                    cpu = {"value": v, "unit": UNIT, "cores": procs, "kind": "reference",
                           "sample": f"{procs} processes x {args.cpu_steps} env-steps of the unmodified reference "
                                     f"(CookingEnvironment.accumulated_step + observe for both agents, reset on episode end; "
                                     f"oracle/_ref behind oracle/refshim), same level / recipe book / action distribution, "
                                     f"{wall:.1f} s wall"}
                except Exception as ex:
                    sys.stderr.write(f"cpu_baseline: the reference arm failed ({ex!r}); reporting the port\n")
            if cpu is None:
                cpu = dict(port)
            else:
                cpu["oracle_port"] = port
            try:
                vc, thr = cpu_port_c_throughput()
                cpu["compiled_port"] = {"value": vc, "unit": UNIT, "threads": thr,
                                        "sample": "4096 envs x 60 steps of oracle/cz_oracle.c (gcc -O2), step + both "
                                                  "observations, all host threads; informational: the reference is Python"}
            except Exception as ex:     # no compiler on the box: the Python port stands alone
                cpu["compiled_port"] = {"unavailable": str(ex)[:120]}
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                "config": workload_config(world, N),
                "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                             "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src,
                             "bytes_per_env_step": bytes_per_env_step,
                             "kernel": ("cz_obs_whole_kernel (+ cz_env_kernel<STEP,dynamics-only> of the next step beside it on a "
                                        "second stream)" if head_pipe else
                                        "cz_obs_whole_kernel (row writer: 82 us of the step) after cz_env_kernel<STEP,dynamics-only> "
                                        "(15 us) on the same stream")},
                "cpu_baseline": cpu,
                "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                        "steps": e2e_steps, "api": "cz_step_host (pinned host buffers, sync per step; four column ranges, the device->host copy of a range "
                               "overlaps the kernels of the next: +0.7 % over one range, CZ_HOST_CHUNKS=1)",
                        "host_link_gbs": (h2d + d2h) * e2e_value / N / 1e9 / world,
                        "limiter": "the host link: the device->host copy of the rows is > 99 % of the call (kernels: 0.11 ms of "
                                   "~11 ms), so chunking the call (done: four ranges) recovers < 1 %; with several GPUs the copies "
                                   "share the host's PCIe root / memory system (host_link_gbs is per GPU)",
                        "numa_node_of_rank0": numa_node},
                "e2e_f32": None if not f32 or "error" in f32 else {
                    "value": f32["e2e_env_steps_per_s"], "unit": UNIT, "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": f32["d2h_bytes_per_step"],
                    "note": "the same call with float32 rows (CZ_STEP_OBS_F32: the float64 rows rounded element-wise, what a "
                            "float32 learner does with the reference's rows): half the bytes over the host link; the "
                            "headline e2e stays float64, the reference's dtype"},
                "gpu_launches": int(launches), "timed_region": how_timed, "clocks": clocks, "cfg3": cfg3, "cfg5": cfg5,
                "generic_tables": generic, "device_policy": cook, "f32_obs": f32,
                "mode": args.mode,
                "mode_note": "sync (default): in-place cz_step, every output ordered on the caller's stream when the call's work "
                             "is done (what a policy that consumes observations uses): dynamics kernel + whole-row TMA writer at "
                             "this batch size; pipelined: cz_step_pipelined, the dynamics of step k+1 on a second stream beside "
                             "the rows of step k (open-loop actions or a policy that reads the state)",
                ("pipelined_step" if not head_pipe else "sync_step"): {
                    "value": other_value, "ms_per_step": ms_other / args.steps,
                    "frac": N * bytes_per_env_step / (ms_other / args.steps / 1e3) / 1e9 / peak,
                    "gpu_launches": int(launches_other), "timed_region": how_other,
                    "note": "the other step mode, same workload, same number of steps"},
                "pipelined_background_dynamics": dict(bg_block, frac=(N * bytes_per_env_step / (bg_block["ms_per_step"] / 1e3) / 1e9 / peak
                                                                      if "ms_per_step" in bg_block else None),
                                                      note="may exceed 1: the roofline peak is a read+write copy bandwidth, the step is "
                                                           "a write stream"),
                "stats": {"episodes_started": float(stats[0]), "recipes_done_now": float(stats[1]),
                          "last_step_return": float(stats[2])}}
        emit(line)
    if world > 1:
        dist.destroy_process_group()


DUMP_ENVS = 8192     # environments whose outputs --dump-outputs writes: 8192 x 2 agents x 278 f64 observations = 36 MB


def dump_outputs(env, out_dir):
    """What the last timed step returned to its caller (observations, rewards, terminated / truncated flags and the info
    fields), as out_dir/<name>.npy, for a fixed seeded sample of DUMP_ENVS environments (every environment when there are
    no more); env_index.npy lists the sampled environments.  Integer outputs are written as float32 (exact below 2**24).
    schedule.npy holds how the environment got there: [warm-up steps, untimed graph steps, timed steps, steps per CUDA
    graph (0: eager launches)]; two runs whose schedules differ (a graph capture that failed on one build) computed
    different steps, and their outputs are not comparable."""
    import torch
    env.wait()
    torch.cuda.synchronize(env.device)
    N = env.num_envs
    pick = np.arange(N) if N <= DUMP_ENVS else np.sort(np.random.default_rng(0).choice(N, DUMP_ENVS, replace=False))
    idx = torch.from_numpy(pick).to(env.device)
    info = env.info()
    out = {"obs": env.obs, "reward": env.reward, "terminated": env.terminated, "truncated": env.truncated,
           "info_t": info["t"], "info_done": info["done"], "info_recipe_done": info["recipe_done"],
           "info_active": info["active"], "info_error_flags": info["error_flags"]}
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "env_index.npy"), pick.astype(np.float64))
    np.save(os.path.join(out_dir, "schedule.npy"), np.array(env._bench_schedule, np.float64))
    for name, t in out.items():
        a = t[idx].cpu().numpy()
        np.save(os.path.join(out_dir, name + ".npy"), a if a.dtype in (np.float64, np.float32) else a.astype(np.float32))


_STDOUT_FD = None


def emit(line):
    """the run's JSON line on the real stdout (see main)"""
    sys.stdout.flush()
    if _STDOUT_FD is not None:
        os.dup2(_STDOUT_FD, 1)
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None)
    ap.add_argument("--warmup", type=int, default=None)
    ap.add_argument("--impl", default="cuda", choices=["cuda", "reference"])
    ap.add_argument("--envs", type=int, default=ENVS_PER_GPU, help="environments per GPU")
    ap.add_argument("--e2e-steps", type=int, default=10)
    ap.add_argument("--cpu-steps", type=int, default=6000, help="oracle env-steps per host process for cpu_baseline")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-cfg3", action="store_true")
    ap.add_argument("--cfg5-envs", type=int, default=262144, help="environments of the mixed-agent-count population (cfg5 block)")
    ap.add_argument("--no-bg", action="store_true", help="skip the eager background-dynamics figure of the pipelined block")
    ap.add_argument("--no-graph", action="store_true", help="time eager launches instead of one CUDA graph of the K steps")
    ap.add_argument("--mode", default="sync", choices=["pipelined", "sync"],
                    help="sync (default, the headline): the in-place step (dynamics kernel, then the whole-row TMA writer, caller's "
                         "stream); pipelined: throughput mode for open-loop action streams, the dynamics of step k+1 run beside "
                         "the observation writes of step k (two kernels, two streams, ping-pong state, cz_pipeline_config)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the outputs of the last one (a fixed sample of rank 0's environments) "
                         "as DIR/<name>.npy, to compare two builds output for output")
    args = ap.parse_args()
    if args.steps is not None and args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "cuda":
        ap.error("--dump-outputs writes the outputs of the CUDA path (--impl cuda)")
    # stdout carries exactly one JSON line: everything libraries print while the run is under way (NCCL's version banner
    # goes to stdout when NCCL_DEBUG is set) is sent to stderr, and the descriptor is handed back for the final print
    sys.stdout.flush()
    global _STDOUT_FD
    _STDOUT_FD = os.dup(1)
    os.dup2(2, 1)
    if args.impl == "reference":
        args.steps = args.steps if args.steps is not None else 6000
        args.warmup = args.warmup if args.warmup is not None else 200
        run_reference_arm(args)
    else:
        args.steps = args.steps if args.steps is not None else 2000
        args.warmup = max(3, args.warmup if args.warmup is not None else 50)
        run_gpu_arm(args)


if __name__ == "__main__":
    main()
