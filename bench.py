#!/usr/bin/env python
"""bench.py -- env-steps/s of the batched StrikeForce tick on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Workload (config.workload = "squad5v5"): Squad 5v5 with NPC spawns under the reference's
shipped macros (squad mates and opponents idle unless USE_AGENT_IN_SQUAD_NPCS, macros.hpp:14;
spawned NPC humans and zombies act every step), levels 1-10 round-robin over arenas, the player
driven by the 28-symbol command alphabet (blocks and portals enabled), 131,072 arenas per GPU (BASELINE.json configs[3]:
1M arenas over 8 GPUs; weak scaling), episodes truncated at 2,048 steps and re-created in the
same call, synthetic seeds and action streams of include/sf_synth.h.  Before timing, the arenas
are spread over episode ages (16 staggered partial resets during the untimed set-up) so that the
timed steps see mid-episode populations, not empty maps.

One step = one sf_step over every arena of the rank.  `value` times K steps with actions already
resident in HBM (CUDA events); `e2e` times the same K steps through sf_step_host with HOST
buffers (pinned actions in, sf_step_out back) inside the timed region.  `roofline` is the step
kernel: algorithmic bytes (summed on the device from the live populations, DESIGN.md) over its
CUDA-event duration against MEASURED_PEAKS.json.  `cpu_baseline` / `--impl reference` time the
UNMODIFIED reference tick engine (oracle/_ref/libsfref.so, one process per arena because the
reference keeps its state in globals) on the box's host cores, on a bounded sample of the same
workload.
"""
import argparse
import json
import multiprocessing as mp
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOAD = dict(workload="squad5v5", mode="Squad", squad_agents=False, level_min=1, level_max=10,
                envs_per_gpu=131072, max_steps=2048, alphabet="28-symbol valid_commands minus '3'",
                l2="state per GPU (3.5 GB) far exceeds the 126 MB L2; no flush needed")
METRIC = "env-steps/sec (bit-exact)"
UNIT = "env-steps/s"


# ----------------------------------------------------------------------------- CPU reference arm

def _ref_worker(args):
    """One process = one arena of the unmodified reference (its state is global)."""
    env, level, n_steps, with_obs, noguard = args
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import sfref
    if noguard:
        sfref.LIB_PATH = sfref.NOGUARD_PATH
    from strikeforce_b200 import config as sfcfg
    caps = [sfcfg.DEFAULT_CAPS[k] for k in ("cap_humans", "cap_zombies", "cap_bullets", "cap_chests", "cap_built",
                                            "cap_portals")]
    sfref.lib()
    t0 = time.perf_counter()
    n, _ = sfref.run_stream(env, sfcfg.MODE_SQUAD, level, n_steps, sfcfg.ACTIONS28.decode(), squad_agents=WORKLOAD["squad_agents"],
                            caps=caps, max_steps=WORKLOAD["max_steps"], with_obs=with_obs)
    return n, time.perf_counter() - t0


def _port_worker(args):
    env, level, n_steps, with_obs, _ = args
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import sfo
    from strikeforce_b200 import config as sfcfg
    from strikeforce_b200 import data as sfdata
    cfg = sfcfg.make_config(sfdata.load_default(), mode=sfcfg.MODE_SQUAD, level_min=level, squad_agents=WORKLOAD["squad_agents"],
                            max_steps=WORKLOAD["max_steps"])
    a = sfo.Arena(cfg)
    t0 = time.perf_counter()
    n, _ = a.run_stream(env, level, n_steps, sfcfg.ACTIONS28, with_obs=with_obs)
    return n, time.perf_counter() - t0


def cpu_reference(steps_per_arena, passes=1, with_obs=False, overhead=False):
    """Times the reference's own CPU implementation on all host cores.  Returns a dict for
    the `cpu_baseline` key.  Each arena plays one full truncated episode cycle per pass, the
    same age mix the GPU arm sees."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import sfref
    cores = os.cpu_count() or 1
    kind = "reference" if sfref.available() else "port"
    worker = _ref_worker if kind == "reference" else _port_worker
    jobs = [(e, 1 + e % 10, steps_per_arena, with_obs, False) for e in range(cores * passes)]
    ctx = mp.get_context("spawn")
    t0 = time.perf_counter()
    with ctx.Pool(cores) as pool:
        res = pool.map(worker, jobs, chunksize=1)
    wall = time.perf_counter() - t0
    total = sum(n for n, _ in res)
    busy = sum(t for _, t in res)
    span = max(t for _, t in res) * passes  # all cores run side by side; process start-up excluded
    out = dict(value=total / span, unit=UNIT, cores=cores, kind=kind, per_core=total / busy,
               sample="%d arenas (one process each, %d at a time) x %d steps of squad5v5 incl. auto-reset; "
                      "%.1f s of stepping, %.1f s wall with process start-up" % (len(jobs), cores, steps_per_arena,
                                                                                span, wall))
    if overhead and kind == "reference" and os.path.exists(sfref.NOGUARD_PATH):
        # what the harness's own checks cost (capacity tracking after every phase, the out-of-bounds scan
        # before update_bull: oracle/ref_harness/harness.cpp): the same arenas with the checks compiled out
        q = max(1024, steps_per_arena // 4)
        with ctx.Pool(cores) as pool:
            r1 = pool.map(worker, [(e, 1 + e % 10, q, with_obs, False) for e in range(cores)], chunksize=1)
        with ctx.Pool(cores) as pool:
            r0 = pool.map(worker, [(e, 1 + e % 10, q, with_obs, True) for e in range(cores)], chunksize=1)
        g1, g0 = sum(n for n, _ in r1) / sum(t for _, t in r1), sum(n for n, _ in r0) / sum(t for _, t in r0)
        out["harness_overhead"] = {"per_core_with_checks": g1, "per_core_without_checks": g0, "slowdown_from_checks": g0 / g1,
                                   "sample": "%d arenas x %d steps each way" % (cores, q)}
    return out


# ----------------------------------------------------------------------------- clocks sampler

class ClockSampler(threading.Thread):
    """SM clock and throttle reasons of one GPU, sampled through NVML while the timed regions run
    (the timed region lasts tens of milliseconds: nvidia-smi, ~100 ms per call, is only the fallback)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        super().__init__(daemon=True)
        self.gpu = gpu_index
        self.sm, self.max_sm, self.reasons = [], [], set()
        self.stop_flag = threading.Event()
        self.nvml = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nvml = pynvml
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(gpu_index)
        except Exception:
            self.nvml = None

    def _sample_nvml(self):
        n = self.nvml
        self.sm.append(float(n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM)))
        self.max_sm.append(float(n.nvmlDeviceGetMaxClockInfo(self.handle, n.NVML_CLOCK_SM)))
        r = n.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle)
        for name, bit in (("hw_slowdown", n.nvmlClocksThrottleReasonHwSlowdown),
                          ("hw_thermal_slowdown", n.nvmlClocksThrottleReasonHwThermalSlowdown),
                          ("sw_thermal_slowdown", n.nvmlClocksThrottleReasonSwThermalSlowdown),
                          ("sw_power_cap", n.nvmlClocksThrottleReasonSwPowerCap)):
            if r & bit:
                self.reasons.add(name)

    def _sample_smi(self):
        out = subprocess.run(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=5).stdout
        for line in out.strip().splitlines():
            r = [x.strip() for x in line.split(",")]
            if len(r) >= 9:
                self.sm.append(float(r[1]))
                self.max_sm.append(float(r[2]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                    if v.lower().startswith("active"):
                        self.reasons.add(name)

    def run(self):
        while not self.stop_flag.is_set():
            try:
                if self.nvml is not None:
                    self._sample_nvml()
                else:
                    self._sample_smi()
            except Exception:
                pass
            self.stop_flag.wait(0.002 if self.nvml is not None else 0.2)

    def summary(self):
        return dict(sm_mhz=statistics.median(self.sm) if self.sm else None, sm_max_mhz=max(self.max_sm) if self.max_sm else None,
                    reasons=sorted(self.reasons), samples=len(self.sm), source="nvml" if self.nvml is not None else "nvidia-smi")


# ----------------------------------------------------------------------------- our arm

def load_traffic(kernel, envs):
    """DRAM bytes per launch of `kernel` from the committed ncu capture, if it was taken at this size."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    try:
        with open(p) as f:
            t = json.load(f)
        return t[kernel]["dram_bytes_per_launch"] if t.get("envs_per_gpu") == envs else None
    except Exception:
        return None


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


DUMP_LIMIT = 64 * 10 ** 6 - 4096  # array bytes of --dump-outputs: under 64 MB with the .npy headers


def step_outputs(sim):
    """What the caller of sim.step reads back after a step, on the host as float64 (exact for int32 and
    for each uint32 half of the 64-bit state hash): per arena its sf_step_out row and its state hash.
    Arenas beyond DUMP_LIMIT are sampled with a fixed seed; `env_ids` says which ones were kept."""
    import numpy as np
    n = sim.n_envs
    keep = np.arange(n)
    per_row = (1 + 8 + 2) * 8
    if n * per_row > DUMP_LIMIT:
        keep = np.sort(np.random.default_rng(0).choice(n, DUMP_LIMIT // per_row, replace=False))
    out = sim.step_out().cpu().numpy()[keep]
    h = sim.state_hash().cpu().numpy()[keep].view(np.uint32).reshape(-1, 2)  # little-endian: low half first
    return {"env_ids": keep.astype(np.float64), "step_out": out.astype(np.float64), "state_hash_lo_hi": h.astype(np.float64)}


def write_outputs(directory, arrays):
    import numpy as np
    os.makedirs(directory, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(directory, name + ".npy"), a)


def run_ours(args):
    import numpy as np
    import torch
    import torch.distributed as dist

    from strikeforce_b200 import config as sfcfg
    from strikeforce_b200 import dist as sfdist
    from strikeforce_b200.sim import BatchedArena

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    E = args.envs
    K, W = args.steps, args.warmup
    table = sfcfg.ACTIONS28
    sim = BatchedArena(E, mode="Squad", level=WORKLOAD["level_min"], level_max=WORKLOAD["level_max"],
                       squad_agents=WORKLOAD["squad_agents"], auto_reset=True, max_steps=WORKLOAD["max_steps"], env_id_base=rank * E)
    A = sim.n_agents
    # ---- untimed set-up: spread the arenas over episode ages
    t = 0
    buckets = 16
    per = max(1, args.prewarm // buckets)
    ids_all = np.arange(E, dtype=np.int32)
    for j in range(buckets):
        for _ in range(per):
            sim.step(sim.synth_actions(t, table))
            t += 1
        if j + 1 < buckets:
            sim.reset(ids_all[ids_all % buckets == j])
    for _ in range(W):
        sim.step(sim.synth_actions(t, table))
        t += 1
    torch.cuda.synchronize()
    pop = sim.population().float().mean(0).tolist()

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident timing: K steps, actions already in HBM
    acts = [sim.synth_actions(t + i, table, out=torch.empty((E, A), dtype=torch.uint8, device=sim.device))
            for i in range(K)]
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    st0 = sim.stats_tensor().clone()
    l0 = sim.launches
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.nvtx.range_push("sf_timed_device")  # `ncu --nvtx --nvtx-include "sf_timed_device/"` sees exactly these launches
    e0.record()
    for i in range(K):
        sim.step(acts[i])
    e1.record()
    torch.cuda.nvtx.range_pop()
    barrier()
    ms_dev = e0.elapsed_time(e1)
    launches = sim.launches - l0
    st1 = sim.stats_tensor().clone()
    dumped = step_outputs(sim) if args.dump_outputs and rank == 0 else None  # the last timed step's results
    t += K
    # ---- end-to-end timing: host actions in, step results out, every step
    acts_h = [a.cpu().pin_memory() for a in
              [sim.synth_actions(t + i, table, out=torch.empty((E, A), dtype=torch.uint8, device=sim.device))
               for i in range(K)]]
    out_h = torch.empty((E, 8), dtype=torch.int32).pin_memory()
    out_np = out_h.numpy().view(sfcfg.STEP_OUT_DTYPE).reshape(E)
    for i in range(min(W, K)):
        sim.step_host(acts_h[i].numpy(), out_np)  # untimed warm-up of the copy path
    st2 = sim.stats_tensor().clone()
    barrier()
    w0 = time.perf_counter()
    e0.record()
    for i in range(K):
        sim.step_host(acts_h[i].numpy(), out_np)
    e1.record()
    barrier()
    ms_e2e_wall = (time.perf_counter() - w0) * 1e3
    ms_e2e = max(e0.elapsed_time(e1), ms_e2e_wall)
    st3 = sim.stats_tensor().clone()
    # ---- second row (SURVEY 8d): step + the player's observation tensor every step, on the device
    obs_row = None
    if not args.no_obs:
        KO = max(2, K // 2)
        obs_buf = torch.empty((E, 1, sfcfg.OBS_CH, sfcfg.OBS_WIN, sfcfg.OBS_WIN), dtype=torch.float32, device=sim.device)
        acts_o = [sim.synth_actions(t + K + i, table, out=acts[i % K]) for i in range(KO)]
        sim.observe(1, out=obs_buf)
        eo = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
        barrier()
        torch.cuda.nvtx.range_push("sf_timed_observe")
        eo[0].record()
        for i in range(KO):
            sim.observe(1, out=obs_buf)
        eo[1].record()
        torch.cuda.nvtx.range_pop()
        for i in range(KO):
            sim.observe(1, out=obs_buf)
            sim.step(acts_o[i])
        eo[2].record()
        barrier()
        ms_obs_only = eo[0].elapsed_time(eo[1])
        ms_both = eo[1].elapsed_time(eo[2])
        # the same observations with the channel innermost (SF_OBS_NHWC: what the policy's convolutions read
        # without a transpose; the reference's own layout is the one above)
        ec = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
        sim.observe(1, out=obs_buf, channels_last=True)
        barrier()
        torch.cuda.nvtx.range_push("sf_timed_observe_nhwc")
        ec[0].record()
        for i in range(KO):
            sim.observe(1, out=obs_buf, channels_last=True)
        ec[1].record()
        torch.cuda.nvtx.range_pop()
        for i in range(KO):
            sim.observe(1, out=obs_buf, channels_last=True)
            sim.step(acts_o[i])
        ec[2].record()
        barrier()
        obs_row = (KO, ms_obs_only, ms_both, ec[0].elapsed_time(ec[1]), ec[1].elapsed_time(ec[2]))
    if rank == 0:
        sampler.stop_flag.set()
        sampler.join()
    # ---- reduce over ranks: max time, summed statistics (the only collective: NCCL all-reduce)
    local_algo = float((st1 - st0)[sfcfg.STAT_NAMES.index("algo_bytes")].item())
    ms_dev = sfdist.max_over_ranks(ms_dev, sim.device)
    ms_e2e = sfdist.max_over_ranks(ms_e2e, sim.device)
    d_dev, d_e2e = sfdist.reduce_stats(st1 - st0), sfdist.reduce_stats(st3 - st2)
    names = sfcfg.STAT_NAMES
    d_dev = dict(zip(names, d_dev.cpu().tolist()))
    d_e2e = dict(zip(names, d_e2e.cpu().tolist()))
    if rank == 0:
        peak, peak_src = load_peaks()
        steps_done = d_dev["steps"] + d_dev["overflows"] + d_dev["ub_guards"]
        value = steps_done / (ms_dev / 1e3)
        e2e_steps = d_e2e["steps"] + d_e2e["overflows"] + d_e2e["ub_guards"]
        achieved = local_algo / (ms_dev / 1e3) / 1e9
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": ms_dev / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "int32", "data": "synthetic (seeded maps/seeds and splitmix64 action streams, include/sf_synth.h)",
            "config": dict(WORKLOAD, envs_per_gpu=E, agents_per_env=A),  # the same dict in both arms
            "setup": {"prewarm_steps": args.prewarm,
                      "mean_population": dict(zip(["humans", "zombies", "bullets", "chests", "built", "portals"],
                                                  [round(x, 2) for x in pop])),
                      "note": "untimed: arenas spread over episode ages before the timed steps"},
            "e2e": {"value": e2e_steps / (ms_e2e / 1e3), "unit": UNIT, "h2d_bytes_per_step": E * A * world,
                    "d2h_bytes_per_step": E * 32 * world, "ms_per_step": ms_e2e / K,
                    "note": "sf_step_host: pinned host actions in, sf_step_out[n] back to the host every step; "
                            "observations are device tensors by contract (the with_observation row) and are not copied"},
            "gpu_launches": launches,
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": load_traffic("sf_step_kernel", E), "traffic_source": "profiles/traffic.json (ncu --set full of one launch of this workload)",
                         "peak_source": peak_src, "kernel": "sf_step_kernel<0>",
                         "algo_bytes_per_launch": local_algo / K,
                         "algo_bytes_per_env_step": local_algo / max(1, K * E),
                         "note": "per GPU (rank 0); algorithmic bytes summed on the device from live populations"},
            "clocks": sampler.summary(),
            "episodes": {k: d_dev[k] for k in ("episodes", "wins", "deaths", "timeouts", "truncated", "overflows",
                                               "ub_guards")},
            "rng_draws_per_env_step": d_dev["rng_draws"] / max(1, steps_done),
        }
        if obs_row is not None:
            KO, ms_obs_only, ms_both, ms_cl_only, ms_cl_both = obs_row
            obs_bytes = E * sfcfg.OBS_LEN * 4
            line["with_observation"] = {
                "note": "rank 0; one fp32 [32,31,31] observation of the player per arena per step, written to HBM",
                "value_step_plus_obs": KO * E / (ms_both / 1e3), "unit": UNIT, "ms_per_step": ms_both / KO,
                "observe_kernel_ms": ms_obs_only / KO,
                "roofline": {"bound": "hbm", "kernel": "sf_observe_kernel", "achieved": obs_bytes / (ms_obs_only / KO / 1e3) / 1e9,
                             "peak": peak, "unit": "GB/s", "frac": obs_bytes / (ms_obs_only / KO / 1e3) / 1e9 / peak,
                             "traffic": load_traffic("sf_observe_kernel", E),
                             "algo_bytes_per_observation": sfcfg.OBS_LEN * 4},
                "channels_last": {
                    "note": "the same values written [31][31][32] per observation (SF_OBS_NHWC, sf_observe_kernel<true>)",
                    "value_step_plus_obs": KO * E / (ms_cl_both / 1e3), "ms_per_step": ms_cl_both / KO,
                    "observe_kernel_ms": ms_cl_only / KO,
                    "roofline": {"bound": "hbm", "kernel": "sf_observe_kernel<NHWC>", "achieved": obs_bytes / (ms_cl_only / KO / 1e3) / 1e9,
                                 "peak": peak, "unit": "GB/s", "frac": obs_bytes / (ms_cl_only / KO / 1e3) / 1e9 / peak,
                                 "traffic": load_traffic("sf_observe_kernel_nhwc", E)}}}
        if world == 1 and not args.no_cpu:
            line["cpu_baseline"] = cpu_reference(args.cpu_steps, overhead=True)
        if dumped is not None:
            write_outputs(args.dump_outputs, dumped)
        print(json.dumps(line))
    sim.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


ROYALE = dict(workload="royale16", mode="Royale (AI Battle Royale, gameplay.hpp:1235), 16 players in 4 teams, the reference's 3x30x100 map",
              envs_per_gpu=32768, max_steps=2048, alphabet="agent actions \"+xzqeawsd\" sampled by the policy",
              policy="AgentModel of bots/bot-0.5/Modules.hpp (random-init weights), fp32, one batched forward per tick",
              l2="16 observations per arena = 64.5 GB per tick per GPU; no flush needed")


def run_royale(args):
    """BASELINE.json configs[4] on one GPU's shard: every tick builds the observations of all 16 players of
    every arena on the device (sf_observe), runs ONE batched AgentModel forward over them, samples the 16
    commands and steps -- nothing leaves the device.  `value` = env-steps/s of that whole tick; rows for
    the step alone and step + observations explain it."""
    import torch
    import torch.distributed as dist

    from strikeforce_b200 import bots, policy
    from strikeforce_b200 import config as sfcfg
    from strikeforce_b200 import dist as sfdist
    from strikeforce_b200.sim import BatchedArena

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(local)
    # the reference network is fp32 (libtorch on the CPU); here the linear layers and GRUs stay fp32 and the
    # convolutions run as cuDNN runs them by default on this GPU (TF32 tensor-core math, fp32 accumulate):
    # strict fp32 convolutions (--strict-fp32) cost 1.04 s per tick instead of 0.107 s (profiles/) and the policy
    # is sampled anyway.
    # The parity tests of the network (tests/test_policy_model.py, test_cpp_host.py) run with TF32 off.
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = not args.strict_fp32
    torch.backends.cudnn.benchmark = True  # no effect on the TF32 path; 4x on strict fp32 (cuDNN's default pick is poor there)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    E = args.envs if args.envs != WORKLOAD["envs_per_gpu"] else ROYALE["envs_per_gpu"]
    K, W = args.steps, args.warmup
    teams = [1, 2, 3, 4] * 4
    P = len(teams)
    sim = BatchedArena(E, mode="Royale", teams=teams, auto_reset=True, max_steps=ROYALE["max_steps"], env_id_base=rank * E)
    t = 0
    for _ in range(min(args.prewarm, 512)):
        sim.step(sim.synth_actions(t, sfcfg.ACTIONS28))
        t += 1
    torch.cuda.synchronize()
    pop = sim.population().float().mean(0).tolist()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, n, warm):
        for _ in range(warm):
            fn()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n):
            fn()
        e1.record()
        barrier()
        return sfdist.max_over_ranks(e0.elapsed_time(e1), sim.device) / n

    acts = [sim.synth_actions(t + i, sfcfg.ACTIONS28, out=torch.empty((E, P), dtype=torch.uint8, device=sim.device))
            for i in range(8)]
    it = iter(range(10 ** 9))
    ms_step = timed(lambda: sim.step(acts[next(it) % len(acts)]), 4 * K, W)
    # the observations are written channel-innermost (SF_OBS_NHWC: same values, [31][31][32] per observation) so
    # that the first convolution reads them as they are; --nchw keeps the reference's [32][31][31]
    # (--strict-fp32 keeps the reference's layout: that is the combination that was measured)
    cl = not args.nchw and not args.strict_fp32
    obs = torch.empty((E, P, sfcfg.OBS_WIN, sfcfg.OBS_WIN, sfcfg.OBS_CH) if cl else
                      (E, P, sfcfg.OBS_CH, sfcfg.OBS_WIN, sfcfg.OBS_WIN), dtype=torch.float32, device=sim.device)
    mask = (1 << P) - 1
    ms_observe = timed(lambda: sim.observe(mask, out=obs, channels_last=cl), 2 * K, W)
    model = policy.AgentModel().to(sim.device)
    agent = policy.PolicyAgent(model, E * P, device=sim.device, seed=1 + rank, chunk=args.policy_chunk, t_initial=0,
                               channels_last=cl)
    custom = bots.Custom(agent, channels_last=cl).prepare(sim)
    actions = torch.empty((E, P), dtype=torch.uint8, device=sim.device)
    l0 = sim.launches

    def tick():
        o = sim.observe(mask, out=obs, channels_last=cl)
        with torch.no_grad():
            idx = agent.predict(o.flatten(0, 1))
        actions.copy_(custom._table[idx].view(E, P))
        sim.step(actions)
        custom.new_games(sim, sim.step_out()[:, 0] != sfcfg.RUNNING)

    ms_tick = timed(tick, K, max(1, min(W, 2)))
    launches = (sim.launches - l0) * K // (K + max(1, min(W, 2)))
    # the public loop (bots.play): the same tick through the plugin surface; only the statistics reach the host
    barrier()
    w0 = time.perf_counter()
    stats = bots.play(sim, custom, K)
    barrier()
    ms_play = sfdist.max_over_ranks((time.perf_counter() - w0) * 1e3, sim.device) / K
    if rank == 0:
        sampler.stop_flag.set()
        sampler.join()
        peak, peak_src = load_peaks()
        obs_bytes = E * P * sfcfg.OBS_LEN * 4
        line = {
            "metric": METRIC, "value": world * E / (ms_tick / 1e3), "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": ms_tick, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int32 (tick), fp32 policy" + ("" if args.strict_fp32 else " with TF32 convolutions (cuDNN default)"),
            "data": "synthetic (seeded matches, random-init policy weights)",
            "config": dict(ROYALE, envs_per_gpu=E, agents_per_env=P, observation_layout="nhwc" if cl else "nchw",
                           **({"mode": ROYALE["mode"].replace("the reference's 3x30x100 map", "a larger map, 3x%dx%d: the reference's embedded in open "
                                                              "ground (SF_GEOMETRY; parity there is pinned against the C oracle only)"
                                                              % (sfcfg.ROWS, sfcfg.COLS))} if sfcfg.GEOMETRY_TAG else {})),
            "setup": {"prewarm_steps": min(args.prewarm, 512),
                      "mean_population": dict(zip(["humans", "zombies", "bullets", "chests", "built", "portals"], [round(x, 2) for x in pop]))},
            "e2e": {"value": world * E / (ms_play / 1e3), "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 128 // max(1, K),
                    "ms_per_step": ms_play,
                    "note": "bots.play: observe -> predict -> step through the plugin surface, wall clock; nothing but the "
                            "final statistics reaches the host (observations arrive as device tensors by contract)"},
            "gpu_launches": launches,
            "rows": {"step_only": {"ms_per_step": ms_step, "env_steps_per_s": world * E / (ms_step / 1e3)},
                     "sixteen_observations": {"ms": ms_observe, "GBps": obs_bytes / (ms_observe / 1e3) / 1e9},
                     "agent_decisions_per_s": world * E * P / (ms_tick / 1e3)},
            "roofline": {"bound": "hbm", "kernel": "sf_observe_kernel", "achieved": obs_bytes / (ms_observe / 1e3) / 1e9, "peak": peak,
                         "unit": "GB/s", "frac": obs_bytes / (ms_observe / 1e3) / 1e9 / peak, "traffic": None, "peak_source": peak_src,
                         "algo_bytes_per_observation": sfcfg.OBS_LEN * 4,
                         "note": "the simulator's dominant kernel of this workload; the tick itself is dominated by the fp32 policy forward (library convolutions)"},
            "clocks": sampler.summary(),
            "episodes": {k2: stats[k2] for k2 in ("episodes", "wins", "deaths", "truncated", "overflows", "ub_guards")},
        }
        print(json.dumps(line))
    sim.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    K, W = args.steps, args.warmup
    world = int(os.environ.get("WORLD_SIZE", "1"))
    # one "step" of this arm = a bounded sample: every host core plays cpu_steps env-steps
    vals, last = [], None
    for i in range(W + K):
        last = cpu_reference(args.ref_steps)
        if i >= W:
            vals.append(last["value"])
    v = sum(vals) / len(vals)
    last["value"] = v
    line = {
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
        "ms_per_step": None, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int32",
        "data": "synthetic (seeded maps/seeds and splitmix64 action streams, include/sf_synth.h)",
        "config": dict(WORKLOAD, envs_per_gpu=args.envs, agents_per_env=1),
        "cpu_baseline": last,
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--envs", type=int, default=WORKLOAD["envs_per_gpu"], help="arenas per GPU")
    ap.add_argument("--prewarm", type=int, default=2048, help="untimed set-up steps (age spreading)")
    ap.add_argument("--cpu-steps", type=int, default=16384, help="env-steps per host core for cpu_baseline")
    ap.add_argument("--ref-steps", type=int, default=8192, help="env-steps per host core per reference-arm step")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-obs", action="store_true", help="skip the step+observation row")
    ap.add_argument("--workload", default="squad5v5", choices=["squad5v5", "royale16"],
                    help="squad5v5 = the headline (BASELINE.json configs[3]); royale16 = configs[4]: 16 players per arena, "
                         "their observations and one batched policy forward every tick (use --steps 3)")
    ap.add_argument("--policy-chunk", type=int, default=32768, help="royale16: observations per forward call")
    ap.add_argument("--strict-fp32", action="store_true", help="royale16: convolutions without TF32 (8x slower)")
    ap.add_argument("--nchw", action="store_true", help="royale16: observations in the reference's [32][31][31] layout "
                                                        "(default: channel innermost, SF_OBS_NHWC)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="squad5v5: after the timed steps, write what the last one computed (rank 0's sf_step_out rows "
                         "and state hashes) as DIR/<name>.npy, float64")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "ours" or args.workload != "squad5v5"):
        ap.error("--dump-outputs records the squad5v5 workload of --impl ours")
    if args.impl == "reference":
        run_reference(args)
    elif args.workload == "royale16":
        run_royale(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
