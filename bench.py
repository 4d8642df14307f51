#!/usr/bin/env python
"""bench.py -- env-steps/sec of the batched PMC mocap-tracking rollout (BASELINE.json configs[1]).

One "step" = one policy step (10 physics sub-steps + mocap + observation + reward + termination + auto-reset)
of every environment of the batch.  Contract: see the task statement / DESIGN.md 7.

    python bench.py --gpus 1 --steps 512 --warmup 32            # our CUDA engine; also reports configs[2] and [4] as sub-results
    python bench.py --gpus 1 --steps 512 --warmup 32 --dump-outputs DIR    # ... and what the last timed step returned, for comparing builds
    python bench.py --impl reference --steps 20 --warmup 3      # CPU arm (oracle port; see DESIGN.md 6)
    python -m torch.distributed.run --nnodes=1 --nproc-per-node 8 --master-addr 127.0.0.1 --master-port 29500 \
        bench.py --gpus 8 ...                                    # env shards, one process per GPU, trajectory gather to rank 0

What the one JSON line holds (N = 1): the PMC headline (`value`, `e2e`, `roofline`, `cpu_baseline`, `on_device_actor_loop`) and
the other single-GPU configurations of BASELINE.json as sub-objects `epmc_8192` (configs[2]) and `sepmc_4096pairs` (configs[4]),
each with its own value / e2e / roofline / on_device_actor_loop (the environmental- / strategic-level policy kernel in the loop).  N > 1: the PMC shards with the [128, N, 223] trajectory hand-over to rank 0 always
measured (`gather`), whatever --steps says.
"""
import argparse
import hashlib
import json
import os

if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
    os.environ["NCCL_DEBUG"] = "WARN"
# stdout carries exactly ONE line, the JSON result: libraries that write to file descriptor 1 on their own (NCCL prints its version
# banner there when a communicator is created) are sent to stderr for the whole run, the result goes to the saved descriptor
_RESULT_OUT = os.fdopen(os.dup(1), "w")
os.dup2(2, 1)
os.environ.setdefault("OMP_WAIT_POLICY", "passive")   # CPU arm: idle OpenMP threads must not spin away the container's CPU quota
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

MU_A = np.array([.0124, -.011, -.0793, -.0125, -.0108, -.0806, .0402, -.0505, -.1956, -.0433, -.0515, -.2156], np.float32)
SIGMA_A = np.array([.0853, .1525, .1747, .0847, .1503, .1766, .1025, .2023, .3701, .1021, .2035, .426], np.float32)
UNROLL = 128                            # example_pmc_train.sh:145
PREROLL = 200                           # untimed steps before anything is measured: the engine is aged into its steady state
                                        # (episodes of mixed age, joint-limit rows present) whatever --warmup says (SURVEY 8d config 2)
METRIC = {"pmc": "env-steps/sec PMC mocap-tracking", "epmc": "env-steps/sec EPMC playground",
          "sepmc": "env-steps/sec SEPMC chase-tag game (one env = one pair of robots, shipped empty arena)"}
WORKLOAD = {"pmc": "4096-env batched PMC mocap-tracking, flat ground, per GPU (BASELINE configs[1])",
            "epmc": "8192-env batched EPMC playground (BASELINE configs[2]), per GPU; --element 3 (default) = corridor with cube steps, 1 = hurdles, "
                    "2 = bars, 0 = the flat joystick arena example_epmc_train.sh ships; the reference has box terrain, no heightfield",
            "sepmc": "2-agent SEPMC chase-tag game, 4096 env-pairs (8192 robots), arena of example_sepmc_train.sh (BASELINE configs[4])"}
# algorithmic bytes per env-step, SURVEY 8(d): PMC 157 words read + 262 written; EPMC with a terrain box list 561 read + 991 written
# (element 0 has no box list: 177 + 991); SEPMC per pair-step 2 x (157 + 262 - 207 + 965) + 40 shared words
ALGO_BYTES = {"pmc": 1676, "epmc": 6208, "epmc_flat": 4672, "sepmc": 9576}
OBS_W = {"pmc": 207, "epmc": 916, "sepmc": 965}
ROBOTS_PER_ENV = {"pmc": 1, "epmc": 1, "sepmc": 2}
ELEMENT = [3]
DUMP_ROWS = 4096                        # --dump-outputs: at most 3 workloads x 4096 rows x 979 float32 columns, < 64 MB in all
KERNEL_SOURCES = ["lifelike_agility_and_play_b200/csrc/llq_step16.cuh", "lifelike_agility_and_play_b200/csrc/llq_kernels.cuh", "lifelike_agility_and_play_b200/csrc/llq_cuda.cu",
                  "lifelike_agility_and_play_b200/csrc/llq_math.cuh"]


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=512)
    ap.add_argument("--warmup", type=int, default=32)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--envs", type=int, default=0, help="robots per GPU (default: 4096 PMC, 8192 EPMC / SEPMC)")
    ap.add_argument("--no-gather", action="store_true", help="N>1: skip the trajectory hand-over to rank 0")
    ap.add_argument("--no-sub", action="store_true", help="skip the epmc_8192 / sepmc_4096pairs sub-results")
    ap.add_argument("--cpu-envs", type=int, default=4096, help="CPU arm: environments per step (default: the same 4096-env batch as the GPU arm)")
    ap.add_argument("--element", type=int, default=3, help="EPMC element_id (0 flat joystick arena, 1 hurdles, 2 bars, 3 cubes)")
    ap.add_argument("--env", default="pmc", choices=["pmc", "epmc", "sepmc"],
                    help="headline workload: pmc = BASELINE configs[1]; epmc = configs[2] (8192 envs); sepmc = configs[4] (4096 pairs; --envs counts robots)")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="write what the last timed step of each workload returned (record = obs | action | reward | done as the step kernel "
                         "writes it into the trajectory slab row, reward, done; with --impl reference: the CPU arm's obs, reward, done) as "
                         "DIR/<workload>_<name>.npy in float32; rank 0's shard; a workload of more than %d robots is stored as a fixed, "
                         "seeded sample of %d rows" % (DUMP_ROWS, DUMP_ROWS))
    a = ap.parse_args()
    ELEMENT[0] = a.element
    if a.envs == 0:
        a.envs = 4096 if a.env == "pmc" else 8192
    return a


def bench_mocap(n_clips=66):
    """The shipped clips packed by tools/statistical_pin.py --stage (LLQ_MOCAP_NPZ) when present, else 66 synthetic clips of the
    shipped dataset's shape."""
    from lifelike_agility_and_play_b200.mocap import synthetic_mocap
    path = os.environ.get("LLQ_MOCAP_NPZ", "")
    if path and os.path.exists(path):
        from lifelike_agility_and_play_b200.mocap import load_packed
        t = load_packed(path)
        return t, "shipped clips packed by mocap.save_packed (%s): %d clips, %d frames" % (os.path.basename(path), len(t.offsets) - 1, len(t.frames))
    return synthetic_mocap(n_clips, seed=0), "66 synthetic clips, 229k frames"


_INPUTS = {}


def synthetic_inputs():
    if not _INPUTS:
        from lifelike_agility_and_play_b200.model.compile_model import load_model_blob
        _INPUTS["blob"] = load_model_blob()
        _INPUTS["mocap"], _INPUTS["mocap_note"] = bench_mocap()
    return _INPUTS["blob"], _INPUTS["mocap"]


def action_pool_np(n, count, seed):
    rng = np.random.default_rng(seed)
    a = MU_A + SIGMA_A * rng.standard_normal((count, n, 12)).astype(np.float32)
    return np.clip(a, -1.0, 1.0).astype(np.float32)


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self._stop_evt, self.proc = index, [], threading.Event(), None

    def run(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q, "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, text=True)
            for line in self.proc.stdout:
                if self._stop_evt.is_set():
                    break
                self.rows.append([c.strip() for c in line.split(",")])
        except Exception:
            pass

    def stop(self):
        self._stop_evt.set()
        if self.proc:
            self.proc.terminate()

    def summary(self):
        sm, mx, reasons = [], 0, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx = max(mx, float(r[1]))
                for nme, v in zip(names, r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(nme)
            except Exception:
                continue
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx or None, "reasons": sorted(reasons),
                "samples": len(sm)}


def bind_to_gpu_numa_node(local_rank):
    """Pin this rank (and the pinned host buffers it allocates afterwards, first touch) to the CPUs of its GPU's NUMA node.
    Eight unpinned ranks across two sockets cost half the end-to-end throughput in round 1 (3.4 MB of D2H per step and GPU
    landing on the far socket for GPUs 4-7).  Returns a short description for the JSON line."""
    try:
        import torch
        bus = None
        try:
            p = torch.cuda.get_device_properties(local_rank)
            bus = "%04x:%02x:%02x.0" % (p.pci_domain_id, p.pci_bus_id, p.pci_device_id)
        except Exception:
            out = subprocess.run(["nvidia-smi", "-i", str(local_rank), "--query-gpu=pci.bus_id", "--format=csv,noheader"],
                                 capture_output=True, text=True, timeout=20).stdout.strip()
            if out:
                dom, rest = out.split(":", 1)
                bus = ("%s:%s" % (dom[-4:], rest)).lower()
        if not bus:
            return {"bound": False, "why": "no PCI bus id"}
        node = int(open("/sys/bus/pci/devices/%s/numa_node" % bus).read().strip())
        if node < 0:
            return {"bound": False, "pci": bus, "why": "numa_node = -1 (single node)"}
        cpus = set()
        for part in open("/sys/devices/system/node/node%d/cpulist" % node).read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        cpus &= os.sched_getaffinity(0)
        if not cpus:
            return {"bound": False, "pci": bus, "numa_node": node, "why": "no allowed CPU on that node"}
        os.sched_setaffinity(0, cpus)
        return {"bound": True, "pci": bus, "numa_node": node, "cpus": len(cpus)}
    except Exception as e:   # affinity is an optimisation: never fail the bench on it
        return {"bound": False, "why": "%s: %s" % (type(e).__name__, e)}


def make_engine(lib_or_none, n, env, **over):
    """Engine for the bench workload on the CUDA library (lib_or_none=None) or a given library (the oracle)."""
    from lifelike_agility_and_play_b200 import _capi as capi
    lib = lib_or_none if lib_or_none is not None else capi.load_cuda_library()
    blob, mocap = synthetic_inputs()
    if env == "epmc":
        from lifelike_agility_and_play_b200.sim_envs.playground_env import INIT_STATE_RUN_0, epmc_engine_config
        erc = {'element_id': ELEMENT[0], 'friction_range': [0.4, 3.0], 'cmd_vary_freq_range': [9999, 10000], 'target_spd_range': [0.5, 3.0],
               'hole_config': {'min_gap_height': 0.25, 'max_gap_height': 0.25}, 'auxiliary_radius': 0.02,
               'disturb_force_config': {'start_time': 0.5, 'interval_time': 1.0, 'duration_time': 0.2, 'horizontal_force': [0, 50], 'vertical_force': [0, 10]}}
        cfg = epmc_engine_config(50.0, 50.0, 0.5, 16, 1000, erc)       # train_scripts/example_epmc_train.sh:88-117
        cfg.update(over)
        eng = capi.VecEngine(lib, n, blob, None, **cfg)
        eng.set_init_state(INIT_STATE_RUN_0)
        return eng
    if env == "sepmc":
        from lifelike_agility_and_play_b200.sim_envs.chase_tag_game_env import sepmc_engine_config
        from lifelike_agility_and_play_b200.sim_envs.playground_env import INIT_STATE_RUN_0
        erc = {'friction_range': [0.4, 3.0],
               'disturb_force_config': {'start_time': 0.5, 'interval_time': 1.0, 'duration_time': 0.2, 'horizontal_force': [0, 50], 'vertical_force': [0, 10]}}
        cfg = sepmc_engine_config(50.0, 50.0, 0.5, 16, 1000, erc)      # train_scripts/example_sepmc_train.sh:94-117
        cfg.update(over)
        eng = capi.VecEngine(lib, n, blob, None, **cfg)
        eng.set_init_state(INIT_STATE_RUN_0)
        return eng
    return capi.VecEngine(lib, n, blob, mocap, **over)


# ------------------------------------------------------------------------------------------------ CPU arm
def _cpu_engine(n_envs, env, threads):
    from oracle import oracle
    eng = make_engine(oracle.load(), n_envs, env, seed=1234, auto_reset=1, num_threads=threads)
    eng.reset()
    return eng


def _cpu_quota():
    """CPUs this container may use: min(hardware threads, cgroup CPU quota).  The GPU boxes expose 128 hardware threads under
    a 16-CPU quota; an OpenMP team wider than the quota burns it in spin-waits and gets throttled (measured: 128 threads ->
    3 k env-steps/s, 16-32 threads -> 150-200 k; tools/cpu_arm_sweep.py)."""
    ncpu = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if q != "max":
            return max(1, min(ncpu, int(np.ceil(float(q) / float(per))))), ncpu
    except Exception:
        pass
    try:
        q = float(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read()); per = float(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
        if q > 0:
            return max(1, min(ncpu, int(np.ceil(q / per)))), ncpu
    except Exception:
        pass
    return ncpu, ncpu


def time_cpu_arm(n_envs, steps, warmup, threads=0, env="pmc", repeats=3):
    """Oracle port of the reference step on the host cores (kind 'port': the reference itself is Python over the pybullet wheel,
    which is not installable here -- DESIGN.md 6).  Fixed configuration, no auto-tune: the same batch as the GPU arm per call,
    one OpenMP thread per CPU of the host's quota.  After a >= 1 s spin-up (OpenMP team up, quota burst spent) and max(3, warmup)
    warm-up calls, `steps` calls are timed `repeats` times; the median is the value, min / max are reported beside it.
    Returns (median env-steps/s, seconds of the median repeat, threads, envs per call, [rates], (obs, reward, done) of the last call)."""
    quota, _ = _cpu_quota()
    th = threads if threads > 0 else quota
    rpe = ROBOTS_PER_ENV[env]
    pool = action_pool_np(n_envs, 8, 5678)
    # the >= 1 s spin-up takes a wall-clock number of steps, so it runs on an engine of its own; the timed engine takes a fixed
    # number of warm-up steps and steps the same states from run to run
    spin = _cpu_engine(n_envs, env, th)
    t_start, k = time.perf_counter(), 0
    while time.perf_counter() - t_start < 1.0:
        spin.step(pool[k % 8]); k += 1
    spin.close()
    eng = _cpu_engine(n_envs, env, th)
    for k in range(max(3, warmup)):
        eng.step(pool[k % 8])
    rates, secs = [], []
    for _ in range(repeats):
        t0 = time.perf_counter()
        for k in range(steps):
            last = eng.step(pool[k % 8])
        dt = time.perf_counter() - t0
        secs.append(dt); rates.append((n_envs // rpe) * steps / dt)
    eng.close()
    order = int(np.argsort(rates)[len(rates) // 2])
    return rates[order], secs[order], th, n_envs, rates, last


def cpu_baseline_obj(val, cores, n, steps, rates):
    q, hw = _cpu_quota()
    return {"value": val, "unit": "env-steps/s", "cores": cores, "kind": "port", "cpu_quota": q, "hw_threads": hw,
            "min": float(min(rates)), "max": float(max(rates)), "repeats": len(rates),
            "sample": "%d envs x %d steps of the same workload, median of %d repeats after a >= 1 s warm-up (oracle/libllq_cpu.so, OpenMP over "
                      "envs, threads = the container's CPU quota, whole batch per call)" % (n, steps, len(rates))}


def run_reference(args, rank):
    if rank != 0:
        return
    n = args.cpu_envs if args.env == "pmc" else args.envs
    val, dt, cores, n, rates, (obs, rew, done) = time_cpu_arm(n, args.steps, args.warmup, env=args.env)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, [(args.env, {"outputs": {"obs": obs, "reward": rew, "done": done.astype(np.float32)}})])
    line = {
        "impl": "reference", "metric": METRIC[args.env], "value": val, "unit": "env-steps/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": WORKLOAD[args.env], "envs_per_gpu": n // ROBOTS_PER_ENV[args.env], "envs_per_step": n,
                   "note": "CPU arm: the oracle port steps the same %d-env batch on the host cores" % n},
        "cpu_baseline": cpu_baseline_obj(val, cores, n, args.steps, rates),
        "e2e": {"value": val, "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), file=_RESULT_OUT, flush=True)


# ------------------------------------------------------------------------------------------------ GPU arm
def source_hash():
    h = hashlib.sha256()
    for f in KERNEL_SOURCES:
        h.update(open(os.path.join(ROOT, f), "rb").read())
    return h.hexdigest()[:16]


def measured_traffic(env_key):
    """DRAM bytes per launch of the dominant kernel from the ncu --set full capture of THIS build: profiles/traffic.json holds
    {"source_hash": ..., "<kernel key>": bytes}; a capture of another build (hash mismatch) is not printed."""
    try:
        t = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
    except Exception:
        return None, "no profiles/traffic.json"
    if t.get("source_hash") != source_hash():
        return None, "profiles/traffic.json is from another build (source hash %s != %s): not reported" % (t.get("source_hash"), source_hash())
    return t.get(env_key), t.get("how", "ncu --set full")


def measure(args, env, n, ctx, headline):
    """Times one workload on this rank's GPU.  Returns a dict of per-rank numbers (milliseconds / counts); rank 0 assembles."""
    import torch
    import torch.distributed as dist
    dev, rank, world, local_rank = ctx["dev"], ctx["rank"], ctx["world"], ctx["local_rank"]
    nu = n // ROBOTS_PER_ENV[env]
    ow = OBS_W[env]
    traj_w = ow + 16                        # obs | action 12 | reward | done | neglogp | value
    eng = make_engine(None, n, env, device=local_rank, seed=1234, auto_reset=1, global_env_offset=rank * n)
    eng.set_option("record", 1)             # the step kernel writes action | reward | done into the slab row itself
    eng.reset()
    POOL = 16
    pool = torch.from_numpy(action_pool_np(n, POOL, 5678 + rank)).to(dev)
    do_gather = headline and world > 1 and not args.no_gather
    from lifelike_agility_and_play_b200.parallel import TrajectoryExchange
    xch = TrajectoryExchange(UNROLL, n, traj_w, dev) if (do_gather or headline) else None
    one_slab = None if xch is not None else torch.zeros((UNROLL, n, traj_w), device=dev, dtype=torch.float32)
    reward = torch.zeros((n,), device=dev, dtype=torch.float32)
    done = torch.zeros((n,), device=dev, dtype=torch.uint8)
    flush = ctx["flush"]
    stream = ctx["stream"].cuda_stream
    state = {"i": 0}

    def one_step():
        i = state["i"]
        t = i % UNROLL
        row = (xch.slab() if xch is not None else one_slab)[t]
        # the fused kernel writes the whole record (observation, action, reward, done) straight into the trajectory slab row
        eng.step_device(pool[i % POOL].data_ptr(), row.data_ptr(), reward.data_ptr(), done.data_ptr(), obs_ld=traj_w, stream=stream)
        state["i"], state["row"] = i + 1, row
        if t == UNROLL - 1 and do_gather:
            xch.hand_over()                 # unroll complete: it travels on the side stream while the next one is stepped

    for _ in range(max(PREROLL, args.warmup)):
        one_step()
    torch.cuda.synchronize()

    sampler = ClockSampler(local_rank) if headline else None
    if sampler:
        sampler.start()
        time.sleep(0.3)
    c0 = eng.counters()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    ev0 = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps)]
    ev1 = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps)]
    wall0 = time.perf_counter()
    for i in range(args.steps):
        flush.fill_(i & 0xFF)                       # L2 flush between timed steps (not timed)
        ev0[i].record()
        one_step()
        ev1[i].record()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    wall = time.perf_counter() - wall0
    step_ms = sum(a.elapsed_time(b) for a, b in zip(ev0, ev1))
    c1 = eng.counters()
    # what the last timed step returned, read before the untimed passes below step the engine again
    outputs = None
    if args.dump_outputs:
        outputs = {"record": state["row"][:, :ow + 14].cpu().numpy(), "reward": reward.cpu().numpy(),
                   "done": done.cpu().numpy().astype(np.float32)}

    # hot (no flush, back-to-back) variant: what a resident rollout loop sees
    h0, h1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    h0.record()
    for i in range(args.steps):
        one_step()
    h1.record()
    torch.cuda.synchronize()
    hot_ms = h0.elapsed_time(h1)
    if sampler:
        sampler.stop()

    # trajectory hand-over of one full [128, N, 223] unroll, always measured at N > 1 (SURVEY 8d config 4 / 8e):
    #   blocking  = post the transfer and wait for it with nothing else running
    #   exposed   = (128 steps with the previous unroll in flight on the side stream) - (128 steps alone)
    gather = None
    if do_gather:
        def timed(fn):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            dist.barrier(); torch.cuda.synchronize()
            a.record(); fn(); b.record()
            torch.cuda.synchronize()
            return a.elapsed_time(b)
        state["i"] = 0
        keep = do_gather
        do_gather = False                                    # the stepping below must not post transfers by itself

        def unroll_alone():
            for _ in range(UNROLL):
                one_step()

        def blocking():
            b = xch.hand_over(); xch.wait(b)

        def unroll_overlapped():
            b = xch.hand_over()
            for _ in range(UNROLL):
                one_step()
            xch.wait(b)
        unroll_alone()
        alone = [timed(unroll_alone) for _ in range(2)]
        block = [timed(blocking) for _ in range(3)]
        over = [timed(unroll_overlapped) for _ in range(2)]
        do_gather = keep
        gather = {"blocking_ms": float(np.median(block)), "unroll_alone_ms": float(min(alone)), "unroll_overlapped_ms": float(min(over)),
                  "exposed_ms": max(0.0, float(min(over)) - float(min(alone))), "bytes_per_rank": xch.bytes_per_rank}

    # dominant kernel alone (events inside the engine, on the launching stream), L2 flushed
    eng.set_option("profile", 1)
    ks, kr = [], []
    for i in range(min(args.steps, 64)):
        flush.fill_(i & 0xFF)
        one_step()
        torch.cuda.synchronize()
        a, b = eng.timing()
        ks.append(a); kr.append(b)
    eng.set_option("profile", 0)
    kern_ms, reset_ms = float(np.mean(ks)), float(np.mean(kr))

    # end-to-end through the public host API (numpy in, numpy out; H2D + D2H inside the timed region)
    # (actions come from pinned host memory, results are read back into pinned host memory: VecEngine.step_pinned)
    e2e_steps = min(args.steps, 128)
    host_pool = action_pool_np(n, 4, 999 + rank)
    act_p, obs_p, rew_p, done_p = eng.pinned_io()
    for i in range(4):
        act_p[...] = host_pool[i % 4]
        eng.step_pinned(act_p, obs_p, rew_p, done_p)
    eng.sync()
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    for i in range(e2e_steps):
        act_p[...] = host_pool[i % 4]               # the policy's output lands in the pinned action buffer
        eng.step_pinned(act_p, obs_p, rew_p, done_p)
        _ = float(rew_p[0])                         # host reads the step's result
    eng.sync()
    e2e_s = time.perf_counter() - t0
    # actors that keep the policy on the device: only reward / done travel back, the observation stays in HBM
    t1 = time.perf_counter()
    for i in range(e2e_steps):
        act_p[...] = host_pool[i % 4]
        eng.step_pinned(act_p, None, rew_p, done_p)
        _ = float(rew_p[0])
    eng.sync()
    e2e_dev_obs_s = time.perf_counter() - t1
    e2e_pageable = None
    if headline:
        # the plain numpy API (pageable buffers, staging copies inside llq_step) for comparison
        out = (np.empty((n, ow), np.float32), np.empty((n,), np.float32), np.empty((n,), np.uint8))
        t2 = time.perf_counter()
        for i in range(32):
            eng.step(host_pool[i % 4], out=out)
        e2e_pageable = nu * 32 / (time.perf_counter() - t2)
    res = {"env": env, "n": n, "nu": nu, "ow": ow, "step_ms": step_ms, "hot_ms": hot_ms, "kern_ms": kern_ms, "reset_ms": reset_ms,
           "e2e_s": e2e_s, "e2e_dev_obs_s": e2e_dev_obs_s, "e2e_steps": e2e_steps, "e2e_pageable": e2e_pageable, "wall": wall,
           "launches": int(c1[4] - c0[4]), "gather": gather, "clocks": sampler.summary() if sampler else None,
           "limit_rows_per_env_substep": float(c1[3] - c0[3]) / max(1, nu * ROBOTS_PER_ENV[env] * args.steps * 10),
           "contact_rows_per_env_substep": float(c1[2] - c0[2]) / max(1, nu * ROBOTS_PER_ENV[env] * args.steps * 10),
           "outputs": outputs}
    if headline:
        res["actor"] = actor_loop(args, eng, n, ow, ctx, pool, reward, done) if (env == "pmc" and world == 1) else None
    if env != "pmc" and world == 1:
        res["actor"] = hier_actor_loop(args, eng, n, ow, ctx, pool, reward, done, strategic=(env == "sepmc"))
    eng.close()
    return res


def actor_loop(args, eng, n, ow, ctx, pool, reward, done):
    """Row f2: the whole actor loop on the device -- policy forward (csrc/llq_policy.cu, random weights of the shipped architecture)
    reads the observation rows in place, writes the actions the next fused step consumes; no host round trip."""
    import torch
    from lifelike_agility_and_play_b200.policy import DevicePolicy
    dev, stream = ctx["dev"], ctx["stream"].cuda_stream
    prng = np.random.default_rng(42)
    shapes = [(1, 135), (1, 135), (1, 72), (1, 72), (207, 256), (256,), (256, 256), (256,), (256, 1), (1,), (207, 256), (256,), (256, 256), (256,),
              (256, 32), (32,), (32, 256), (135, 64), (64,), (32, 32), (32,), (96, 256), (256,), (256, 256), (256,), (256, 12), (12,), (1, 12)]
    wts = [(prng.standard_normal(sh) / np.sqrt(sh[0] if len(sh) == 2 and sh[0] > 1 else 1.0)).astype(np.float32) for sh in shapes]
    wts[1] = np.abs(wts[1]) + 0.5; wts[3] = np.abs(wts[3]) + 0.5
    wts[25] *= 0.05                                        # small actions, like a trained policy's
    pol = DevicePolicy(wts, device=ctx["local_rank"])
    eng.set_option("record", 0)
    obs_t = torch.zeros((n, ow), device=dev, dtype=torch.float32)
    act_t = torch.zeros((n, 12), device=dev, dtype=torch.float32)
    eng.step_device(pool[0].data_ptr(), obs_t.data_ptr(), reward.data_ptr(), done.data_ptr(), obs_ld=ow, stream=stream)

    def actor_step():
        pol.forward(obs_t.data_ptr(), ow, n, act_t.data_ptr(), None, stream)
        eng.step_device(act_t.data_ptr(), obs_t.data_ptr(), reward.data_ptr(), done.data_ptr(), obs_ld=ow, stream=stream)
    for i in range(8):
        actor_step()
    torch.cuda.synchronize()
    a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a0.record()
    for i in range(args.steps):
        actor_step()
    a1.record()
    torch.cuda.synchronize()
    actor_ms = a0.elapsed_time(a1)
    p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    p0.record()
    for i in range(64):
        pol.forward(obs_t.data_ptr(), ow, n, act_t.data_ptr(), None, stream)
    p1.record()
    torch.cuda.synchronize()
    val_t = torch.zeros((n,), device=dev, dtype=torch.float32)
    nlp_t = torch.zeros((n,), device=dev, dtype=torch.float32)
    q0, q1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    q0.record()
    for i in range(64):
        pol.forward_ex(obs_t.data_ptr(), ow, n, act_t.data_ptr(), None, val_t.data_ptr(), nlp_t.data_ptr(), 1, i, stream)
    q1.record()
    torch.cuda.synchronize()
    out = {"value": n * args.steps / (actor_ms * 1e-3), "unit": "env-steps/s", "ms_per_step": actor_ms / args.steps,
           "policy_kernel_ms": p0.elapsed_time(p1) / 64, "policy_kernel_ms_with_value_head_and_sampling": q0.elapsed_time(q1) / 64,
           "policy": "PMC net 207-256-256-32 VQ(256) + 135/32-96-256-256-12, 3xTF32 mma.sync (fp32-level accuracy), random weights",
           "note": "policy forward + fused env step, observations and actions stay in HBM (hot L2, no flush)"}
    pol.close()
    return out


def hier_actor_loop(args, eng, n, ow, ctx, pool, reward, done, strategic):
    """Row f2 for the environmental / strategic level: csrc/llq_policy_hier.cu (random weights of the shipped architecture) reads the
    observation rows in place, keeps its LSTM states on the device, resets them from the engine's own done flags."""
    import torch
    from lifelike_agility_and_play_b200.policy_epmc import DeviceHierPolicy, random_weights
    dev, stream = ctx["dev"], ctx["stream"].cuda_stream
    wts = random_weights(strategic, seed=42)
    li = 150 if strategic else 100                           # last decoder layer: small actions, like a trained policy's
    wts[li - 1] = wts[li - 1] * 0.05
    pol = DeviceHierPolicy(wts, device=ctx["local_rank"])
    eng.set_option("record", 0)
    obs_t = torch.zeros((n, ow), device=dev, dtype=torch.float32)
    act_t = torch.zeros((n, 12), device=dev, dtype=torch.float32)
    st_t = torch.zeros((n, pol.state_dim), device=dev, dtype=torch.float32)
    eng.step_device(pool[0].data_ptr(), obs_t.data_ptr(), reward.data_ptr(), done.data_ptr(), obs_ld=ow, stream=stream)

    def actor_step():
        pol.forward(obs_t.data_ptr(), ow, n, done.data_ptr(), st_t.data_ptr(), act_t.data_ptr(), None, None, stream)
        eng.step_device(act_t.data_ptr(), obs_t.data_ptr(), reward.data_ptr(), done.data_ptr(), obs_ld=ow, stream=stream)
    for i in range(8):
        actor_step()
    torch.cuda.synchronize()
    a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a0.record()
    for i in range(args.steps):
        actor_step()
    a1.record()
    torch.cuda.synchronize()
    actor_ms = a0.elapsed_time(a1)
    p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    p0.record()
    for i in range(32):
        pol.forward(obs_t.data_ptr(), ow, n, done.data_ptr(), st_t.data_ptr(), act_t.data_ptr(), None, None, stream)
    p1.record()
    torch.cuda.synchronize()
    units = n // 2 if strategic else n
    out = {"value": units * args.steps / (actor_ms * 1e-3), "unit": "pair-steps/s" if strategic else "env-steps/s", "ms_per_step": actor_ms / args.steps,
           "policy_kernel_ms": p0.elapsed_time(p1) / 32, "policy_rows": n,
           "policy": ("strategic-level net (heading controller + code controller + frozen decoder)" if strategic else
                      "environmental-level net (conv encoders, layer-norm LSTM, 256-way code, frozen decoder)") +
                     ", fp32 CUDA cores, one CTA per row, random weights (csrc/llq_policy_hier.cu)",
           "note": "policy forward + fused env step; observations, LSTM states and actions stay in HBM (hot L2, no flush)"}
    pol.close()
    return out


def dump_outputs(path, results):
    """--dump-outputs: DIR/<workload>_<name>.npy for each (workload, per-rank result) pair; the sampled rows depend on the row count only."""
    os.makedirs(path, exist_ok=True)
    for key, r in results:
        n = len(r["outputs"]["reward"])
        rows = np.sort(np.random.default_rng(0).choice(n, DUMP_ROWS, replace=False)) if n > DUMP_ROWS else slice(None)
        for name, a in r["outputs"].items():
            np.save(os.path.join(path, "%s_%s.npy" % (key, name)), np.ascontiguousarray(a[rows], np.float32))


def kernel_name(env):
    inst = {"pmc": 0, "epmc": 1 if ELEMENT[0] == 0 else 3, "sepmc": 2}[env]
    return "llq_step16_kernel<%d>" % inst


def assemble(args, r, world, peak, peak_src, reduce_max):
    """Whole-job numbers of one workload from the per-rank result r (times are max over ranks)."""
    env, nu, n, ow = r["env"], r["nu"], r["n"], r["ow"]
    step_ms, hot_ms, kern_ms, reset_ms, e2e_s, e2e_dev_obs_s = reduce_max([r["step_ms"], r["hot_ms"], r["kern_ms"], r["reset_ms"], r["e2e_s"], r["e2e_dev_obs_s"]])
    g = r["gather"]
    exposed = 0.0
    if g is not None:
        g = dict(g)
        g["blocking_ms"], g["unroll_alone_ms"], g["unroll_overlapped_ms"], g["exposed_ms"] = reduce_max(
            [g["blocking_ms"], g["unroll_alone_ms"], g["unroll_overlapped_ms"], g["exposed_ms"]])
        g["exposed_frac_of_unroll"] = g["exposed_ms"] / g["unroll_alone_ms"]
        g["how"] = ("grouped ncclSend/ncclRecv (torch batch_isend_irecv) of the finished [128, N_local, %d] slab on a side stream, ping-pong slabs; "
                    "exposed = 128 steps with the transfer in flight - 128 steps alone; amortised into `value` as exposed_ms per 128 steps" % (ow + 16))
        exposed = g["exposed_ms"] * args.steps / UNROLL
    total_ms = step_ms + exposed
    total = nu * world * args.steps
    akey = "epmc_flat" if (env == "epmc" and ELEMENT[0] == 0) else env
    achieved = ALGO_BYTES[akey] * nu / (kern_ms * 1e-3) / 1e9
    traffic, traffic_note = measured_traffic(kernel_name(env))
    out = {
        "metric": METRIC[env], "value": total / (total_ms * 1e-3), "unit": "env-steps/s", "ms_per_step": total_ms / args.steps,
        "value_hot_l2": total / (hot_ms * 1e-3), "value_no_gather": total / (step_ms * 1e-3),
        "robot_steps_per_s": ROBOTS_PER_ENV[env] * total / (total_ms * 1e-3),
        "e2e": {"value": nu * world * r["e2e_steps"] / e2e_s, "unit": "env-steps/s", "h2d_bytes_per_step": n * 12 * 4,
                "d2h_bytes_per_step": n * (ow * 4 + 4 + 1), "steps": r["e2e_steps"],
                "api": "VecEngine.step_pinned(numpy over page-locked memory) -> llq_step_ex(LLQ_IO_PINNED)",
                "value_device_resident_obs": nu * world * r["e2e_steps"] / e2e_dev_obs_s,
                "device_resident_obs_note": "same call with obs=None: reward / done travel back (5 B per env), the observation stays in HBM for an on-device policy"},
        "gpu_launches": r["launches"],
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                     "traffic_note": traffic_note, "kernel": kernel_name(env), "kernel_ms": kern_ms, "reset_kernel_ms": reset_ms,
                     "algorithmic_bytes_per_env_step": ALGO_BYTES[akey], "peak_source": peak_src,
                     "note": "latency/issue bound by design (SURVEY 7): ~2e5 flop per 1.7 kB of state; see profiles/"},
        "workload_stats": {"limit_rows_per_robot_substep": r["limit_rows_per_env_substep"], "contact_rows_per_robot_substep": r["contact_rows_per_env_substep"]},
    }
    if r["e2e_pageable"] is not None:
        out["e2e"]["value_pageable_numpy_api"] = r["e2e_pageable"] * world
    if g is not None:
        out["gather"] = g
    return out


def main():
    args = parse()
    rank = int(os.environ.get("RANK", 0))
    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    if args.impl == "reference":
        return run_reference(args, rank)

    import torch
    import torch.distributed as dist

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    numa = bind_to_gpu_numa_node(local_rank)       # before any pinned allocation
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    # everything below runs on one explicit (non-default) stream: the engine launches on it, the CUDA events are
    # recorded on it (torch.cuda.Event only sees torch's current stream)
    bench_stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(bench_stream)
    assert bench_stream.cuda_stream != 0
    ctx = {"dev": dev, "rank": rank, "world": world, "local_rank": local_rank, "stream": bench_stream,
           "flush": torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)}          # > 126 MB L2

    def reduce_max(vals):
        t = torch.tensor(vals, device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return [float(x) for x in t.tolist()]

    head = measure(args, args.env, args.envs, ctx, True)
    subs = {}
    if args.env == "pmc" and not args.no_sub:
        # BASELINE configs[2]: 8192 EPMC envs per GPU (weak); configs[4]: 4096 chase-tag pairs in total, sharded over the ranks
        # (2 x 2048 pairs at N = 2 is exactly configs[4]; strong scaling, noted in the sub-object)
        subs["epmc_8192"] = measure(args, "epmc", 8192, ctx, False)
        pairs_per_rank = max(1, 4096 // world)
        subs["sepmc_4096pairs"] = measure(args, "sepmc", 2 * pairs_per_rank, ctx, False)

    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6650 GB/s (B200_PROFILING.md)"
    h = assemble(args, head, world, peak, peak_src, reduce_max)
    sub_out = {k: assemble(args, v, world, peak, peak_src, reduce_max) for k, v in subs.items()}
    numa_all = [numa]
    if world > 1:
        numa_all = [None] * world
        dist.all_gather_object(numa_all, numa)
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    if args.dump_outputs:
        dump_outputs(args.dump_outputs, [(args.env, head)] + list(subs.items()))
    env = args.env
    do_gather = world > 1 and not args.no_gather
    synthetic_inputs()
    line = {
        "metric": h["metric"], "value": h["value"], "unit": "env-steps/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": h["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD[env] + ("; sharded as in configs[3]" if world > 1 else ""),
                   "element_id": args.element if env == "epmc" else None, "envs_per_gpu": head["nu"], "global_envs": head["nu"] * world,
                   "robots_per_gpu": head["n"], "substeps": 10, "solver_iters": 10,
                   "mocap": _INPUTS.get("mocap_note") if env == "pmc" else None,
                   "auto_reset": True, "prioritized_sample_factor": 3.0 if env == "pmc" else None,
                   "actions": "N(mu_a, sigma_a) clipped +-1, device resident",
                   "preroll_steps": max(PREROLL, args.warmup),
                   "preroll_note": "untimed steps before the timed region whatever --warmup says: steady-state episode mix (SURVEY 8d)",
                   "l2": "flushed (256 MiB write) between timed steps; per-step CUDA events summed",
                   "record": "the step kernel writes obs | action | reward | done of every record into the [128, N, %d] trajectory slab row" % (head["ow"] + 16),
                   "numa": numa_all,
                   "parallelism": "env shards x%d%s" % (world, ", finished [128,N,obs+16] slabs handed to rank 0 by grouped NCCL send/recv on a side stream, "
                                                               "overlapped with the next unroll" if do_gather else "")},
        "value_hot_l2": h["value_hot_l2"], "value_no_gather": h["value_no_gather"],
        "gather_ms_total": (h["gather"]["exposed_ms"] * args.steps / UNROLL) if "gather" in h else 0.0,
        "wall_s_timed_region": head["wall"],
        "e2e": h["e2e"], "gpu_launches": h["gpu_launches"], "roofline": h["roofline"], "workload_stats": h["workload_stats"],
        "clocks": head["clocks"],
    }
    if "gather" in h:
        line["gather"] = h["gather"]
    if head.get("actor"):
        line["on_device_actor_loop"] = head["actor"]
    for k, v in sub_out.items():
        if subs[k].get("actor"):
            v["on_device_actor_loop"] = subs[k]["actor"]
        v["config"] = {"workload": WORKLOAD["epmc" if k.startswith("epmc") else "sepmc"], "envs_per_gpu": subs[k]["nu"], "robots_per_gpu": subs[k]["n"],
                       "scaling": "weak" if k.startswith("epmc") else "strong (4096 pairs in total over %d GPU%s)" % (world, "s" if world > 1 else ""),
                       "element_id": ELEMENT[0] if k.startswith("epmc") else None, "preroll_steps": max(PREROLL, args.warmup)}
        line[k] = v
    if world == 1:
        cn = args.cpu_envs if env == "pmc" else args.envs
        cval, cdt, cores, cne, rates, _ = time_cpu_arm(cn, 32, 3, env=env)
        line["cpu_baseline"] = cpu_baseline_obj(cval, cores, cne, 32, rates)
    print(json.dumps(line), file=_RESULT_OUT, flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
