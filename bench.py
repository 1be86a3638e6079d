#!/usr/bin/env python
"""bench.py -- agent-steps/sec of the batched gym-macm step on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W]            # this repo's CUDA path
    python bench.py --impl reference [--gpus N] --steps K --warmup W   # the CPU path, timed beside it

Workload (BASELINE.json configs[1]): cm-flock-v0, 64 agents x 4096 envs per GPU, linear reward,
discrete U{0,1,2}^3 actions, initial states drawn from the reference's distributions.  One "step"
is one Flock.step for all 4096 envs = one kernel launch.  The footprint of one batch (~20 MB)
fits in the 126 MB L2, so the timed loop rotates over ROT independent batches (> 2x L2 in
total): every step's inputs come from HBM.

The headline spreads the rotation's independent batches over two streams (a batch keeps its stream): one
batch's last envs -- a few worlds with long contact islands -- finish while the next batch's blocks take over
the SMs.  --steps is the number of timed steps; --windows splits them into windows and the per-rank median of
the time per step is taken.  --dump-outputs DIR writes what the last timed step returned (obs, rewards, done,
nearest-agent ids, collided flags of the batch it stepped) as .npy files: the inputs are seeded, so two builds
run with the same arguments can be compared output for output.

N > 1 (torchrun, one rank per GPU): each rank owns its own 4096 envs (weak scaling); envs are
independent, so the data path has no collective.  Legs beside the headline: the same steps on one stream,
an isolated launch, macm_rollout, BASELINE configs 3 / 4 / 5 (16M-agent point), and with N > 1 the
learner-side exchange of config 5 both ways (step kernel storing into the learner's memory over NVLink,
and an NCCL all-gather).
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "gym-macm_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

N_AGENTS, N_ENVS = 64, 4096
WORKLOAD = "cm-flock-v0 64 agents x 4096 envs per GPU, linear reward, discrete random actions"
METRIC, UNIT = "agent_steps_per_sec", "agent-steps/s"


def measured_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured"
    except Exception:
        return 6650.0, "fallback"


_NVML_SAMPLER = r"""
import sys, time
import pynvml as N
N.nvmlInit()
h = N.nvmlDeviceGetHandleByIndex(int(sys.argv[1]))
mx = N.nvmlDeviceGetMaxClockInfo(h, N.NVML_CLOCK_SM)
get = getattr(N, "nvmlDeviceGetCurrentClocksEventReasons", None) or N.nvmlDeviceGetCurrentClocksThrottleReasons
while True:
    sm = N.nvmlDeviceGetClockInfo(h, N.NVML_CLOCK_SM)
    r = get(h)
    sys.stdout.write("%.6f,%d,%d,%d\n" % (time.time(), sm, mx, r))
    sys.stdout.flush()
    time.sleep(0.001)
"""


class ClockSampler(object):
    """SM clock and throttle reasons while the timed region runs: an NVML poller in its own process (about one
    sample per millisecond, no GIL shared with the launch loop); `nvidia-smi -lms` when pynvml is missing."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")
    BITS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap",
            0x80: "hw_power_brake_slowdown"}

    def __init__(self, index):
        self.rows, self.proc, self.kind = [], None, None
        for kind, cmd in (("nvml", [sys.executable, "-c", _NVML_SAMPLER, str(index)]),
                          ("nvidia-smi", ["nvidia-smi", "-i", str(index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "20"])):
            try:
                self.proc = subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
                self.kind = kind
                self.th = threading.Thread(target=self._read, daemon=True)
                self.th.start()
                t_end = time.time() + 5.0          # wait for the first sample (NVML init)
                while not self.rows and self.proc.poll() is None and time.time() < t_end:
                    time.sleep(0.01)
                if self.rows:
                    break
                self.proc.kill()
                self.proc = None
            except Exception:
                self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def _parse(self, t_host, line):
        f = [x.strip() for x in line.split(",")]
        if self.kind == "nvml":
            bits = int(f[3])
            return float(f[0]), float(f[1]), float(f[2]), [nm for b, nm in self.BITS.items() if bits & b]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        return t_host, float(f[0]), float(f[1]), [nm for nm, v in zip(names, f[3:7]) if v.lower().startswith("active")]

    def stop(self, t0, t1):
        """Samples taken inside [t0, t1]; if the region was too short to hold three of them, the nearest ones
        taken under the same load (the warm-up steps run right before it) are added and counted separately."""
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no clock sampler available"], "samples": 0}
        time.sleep(0.03)
        self.proc.kill()
        got = []
        for th, line in list(self.rows):
            try:
                got.append(self._parse(th, line))
            except Exception:
                continue
        inside = [g for g in got if t0 <= g[0] <= t1]
        near = []
        if len(inside) < 3:
            near = sorted((g for g in got if g not in inside and t0 - 0.25 <= g[0] <= t1 + 0.002), key=lambda g: -g[0])[:8]
        use = inside + near
        reasons = sorted(set(r for g in use for r in g[3]))
        return {"sm_mhz": statistics.median([g[1] for g in use]) if use else None,
                "sm_max_mhz": use[0][2] if use else None, "reasons": reasons, "samples": len(inside),
                "samples_warmup": len(near), "sampler": self.kind}


def b_alg_per_agent_step(c_bar, T, N):
    # SURVEY.md 8(d): state r/w 40+40, action 4, target index 1, obs 20, reward 4 = 109 B,
    # + 32 B per live contact per agent (16-byte record read + written), + amortised targets/done
    return 109.0 + 32.0 * c_bar + (8.0 * T + 1.0) / N


def random_state(rng, E, N, T, spread=20.0):
    """The reference's initial distributions (mvmnt.py:48-52,62-64), as float64 draws."""
    import numpy as np
    pos = spread * (rng.random((E, N, 2)) - 0.5)
    ang = rng.uniform(-1, 1, (E, N)) * np.pi
    ta = 2 * np.pi * rng.random((E, T))
    td = 25 + rng.random((E, T)) * 35
    return pos, ang, np.stack([td * np.cos(ta), td * np.sin(ta)], -1)


def cpu_oracle_rate(n_envs, n_threads, budget_s, seed=1234):
    """agent-steps/s of the CPU oracle (restatement, not pybox2d) on `n_threads` host threads."""
    import numpy as np
    from oracle import oracle
    rng = np.random.default_rng(seed)
    pos, ang, tg = random_state(rng, n_envs, N_AGENTS, 1)
    ref = oracle.OracleBatch(n_envs, n_agents=N_AGENTS, n_targets=1, reward_mode=1,
                             damping_model=DAMPING_CODE[default_damping()])
    ref.reset(pos, ang, targets=tg)
    acts = rng.integers(0, 3, (8, n_envs, N_AGENTS, 3)).astype(np.int32)
    for k in range(2):
        ref.flock_step(acts[k], n_threads)
    steps, t0 = 0, time.perf_counter()
    while True:
        ref.flock_step(acts[steps % 8], n_threads)
        steps += 1
        el = time.perf_counter() - t0
        if el >= budget_s:
            break
    return n_envs * N_AGENTS * steps / el, steps, el


def pybox2d_probe(seconds=0.0):
    """oracle/pybox2d_probe.py in a subprocess (clean sys.path): is a real Box2D importable, what do the
    discriminators select, and -- with `seconds` -- how fast is the reference's own Flock.step loop."""
    try:
        out = subprocess.run([sys.executable, os.path.join(ROOT, "oracle", "pybox2d_probe.py"), "--time", str(seconds)],
                             capture_output=True, text=True, timeout=60 + 4 * seconds, env={**os.environ, "PYTHONPATH": ROOT})
        return json.loads(out.stdout.strip().splitlines()[-1])
    except Exception as ex:
        return {"available": False, "why": "probe failed: %r" % (ex,)}


def run_reference(args, rank, world):
    """--impl reference: the reference's CPU implementation of the path.  The probe looks for a real pybox2d first
    (kind "pybox2d": the reference's own Flock.step loop); without one -- this image has no wheel and no network --
    it is the oracle port on every host thread (kind "port")."""
    if rank != 0:
        return
    import numpy as np
    from oracle import oracle
    oracle.build()
    cores = len(os.sched_getaffinity(0))
    probe = pybox2d_probe(seconds=8.0)
    real = probe.get("reference_loop") if probe.get("available") else None
    # a bounded sample of the 4096-env batch per step: 64 envs per host thread, so that starting and joining the
    # worker threads (once per step) stays below a tenth of the step
    sample_envs = min(N_ENVS, 64 * cores)
    rng = np.random.default_rng(1234)
    pos, ang, tg = random_state(rng, sample_envs, N_AGENTS, 1)
    ref = oracle.OracleBatch(sample_envs, n_agents=N_AGENTS, n_targets=1, reward_mode=1,
                             damping_model=DAMPING_CODE[default_damping()])
    ref.reset(pos, ang, targets=tg)
    acts = rng.integers(0, 3, (16, sample_envs, N_AGENTS, 3)).astype(np.int32)
    for k in range(args.settle + args.warmup):      # the same 64 settle steps after the spawn as the GPU arm, untimed
        ref.flock_step(acts[k % 16], cores)
    t0 = time.perf_counter()
    for k in range(args.steps):
        ref.flock_step(acts[k % 16], cores)
    el = time.perf_counter() - t0
    val = sample_envs * N_AGENTS * args.steps / el
    sample = "%d of the %d envs per step (x%d agents), %d steps after %d settle steps, oracle port on %d threads" % (
        sample_envs, N_ENVS, N_AGENTS, args.steps, args.settle, cores)
    kind = "port"
    if real and "agent_steps_per_sec" in real:
        # the real thing: pybox2d + the reference's Python host, single process (it has no batch axis)
        kind, val, cores = "pybox2d", float(real["agent_steps_per_sec"]), 1
        sample = "the reference's Flock.step loop, 1 env x %d agents, %d steps in %.1f s, single process" % (
            real["n_agents"], real["steps"], real["seconds"])
        el = args.steps * N_ENVS * N_AGENTS / val
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * el / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "sample": sample,
                   "note": "pybox2d is not installable here; CPU restatement (oracle/), not pybox2d" if kind == "port"
                           else "pybox2d + the reference's Python host",
                   "pybox2d_probe": {k: probe.get(k) for k in ("available", "why", "damping_model", "box2d_version") if k in probe}},
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


DAMPING_CODE = {"taylor": 0, "pade": 1}


def default_damping():
    from gym_macm.settings import flockSettings
    return flockSettings().damping_model


class Timer(object):
    """Device timing of step sequences: K steps in all, split into windows as evenly as possible, each window
    bracketed by a barrier over the ranks and a device synchronisation on both sides and timed with CUDA events on
    the stream the steps are enqueued from (side streams fork after the start event and join before the stop
    event).  A rank's figure is the MEDIAN over its windows of the time per step; the job's figure is the MAX over
    the ranks."""

    def __init__(self, torch, dist, dev, world):
        self.torch, self.dist, self.dev, self.world = torch, dist, dev, world
        self.main = torch.cuda.current_stream(dev)

    def max_over_ranks(self, x):
        if self.world > 1:
            t = self.torch.tensor([x], device=self.dev, dtype=self.torch.float64)
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
            return float(t.item())
        return x

    def windows(self, issue, K, n_windows, streams=(), k0=0, after=None):
        """Issue steps k0 .. k0 + K - 1; returns (ms per step, [ms of each window], next k)."""
        torch = self.torch
        n_windows = max(1, min(n_windows, K))
        sizes = [K // n_windows + (w < K % n_windows) for w in range(n_windows)]
        ms, k = [], k0
        for n in sizes:
            torch.cuda.synchronize()
            if self.world > 1:
                self.dist.barrier()
                torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for st in streams:
                st.wait_stream(self.main)      # every stream starts after the start event ...
            for j in range(n):
                issue(k)
                k += 1
            for st in streams:
                self.main.wait_stream(st)      # ... and the stop event waits for all of them
            if after is not None:
                after()
            e1.record()
            torch.cuda.synchronize()
            ms.append(e0.elapsed_time(e1))
        med = statistics.median(m / n for m, n in zip(ms, sizes))
        return self.max_over_ranks(med), ms, k


DUMP_LIMIT = 64 << 20   # bytes written by --dump-outputs in all


def dump_outputs(path, batch):
    """The per-step outputs of `batch` (what a caller of the stepped batch reads) as DIR/<name>.npy: float outputs
    in float32, integer ones in float64 (exact).  Past DUMP_LIMIT a fixed, seeded sample of envs is written;
    env_index.npy names the envs written either way."""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    out = {}
    for name in batch.engine.OUTPUTS:
        a = batch.state[name].cpu().numpy()
        out[name] = a.astype(np.float32 if a.dtype.kind == "f" else np.float64)
    E = batch.engine.E
    per_env = sum(a.nbytes for a in out.values()) // E + 8
    keep = np.arange(E)
    if per_env * E > DUMP_LIMIT:
        keep = np.sort(np.random.default_rng(0).choice(E, (DUMP_LIMIT - 4096) // per_env, replace=False))   # 4 KB: .npy headers
    out["env_index"] = keep.astype(np.float64)
    for name, a in out.items():
        np.save(os.path.join(path, name + ".npy"), a if name == "env_index" else a[keep])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2000)
    ap.add_argument("--warmup", type=int, default=50)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--rot", type=int, default=16, help="independent batches rotated through (L2 eviction)")
    ap.add_argument("--envs", type=int, default=N_ENVS)
    ap.add_argument("--no-numa", action="store_true", help="do not bind the ranks to their GPU's NUMA node")
    ap.add_argument("--rollout", type=int, default=32, help="steps per launch of the macm_rollout leg (0 = skip it)")
    ap.add_argument("--streams", type=int, default=2,
                    help="streams the independent batches of the rotation are spread over (a batch keeps its stream); "
                         "2 = a batch's last envs finish while the next batch starts")
    ap.add_argument("--windows", type=int, default=1,
                    help="timed windows the --steps steps are split into (the median time per step is reported)")
    ap.add_argument("--no-legs", action="store_true", help="headline + e2e only (no other configs, no exchange legs)")
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--e2e-steps", type=int, default=240)
    ap.add_argument("--e2e-depth", type=int, default=3, help="independent batches in flight on the host-buffer path")
    ap.add_argument("--policy", default="random", choices=["random", "flock"])
    ap.add_argument("--settle", type=int, default=64, help="untimed steps per batch after the random spawn")
    ap.add_argument("--max-touching", type=int, default=0, help="experiment: capacity of the touching-contact stage (0 = default)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the outputs of the last one to DIR/<name>.npy (float32/float64)")
    args = ap.parse_args()
    if args.steps < 1 or args.windows < 1:
        ap.error("--steps and --windows must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the CUDA path's outputs; --impl reference has none to write")

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if args.warmup < 3:
        args.warmup = 3

    import numpy as np
    import torch
    import torch.distributed as dist
    import gym_macm

    numa_cpus = None
    if world > 1 and not args.no_numa:
        from gym_macm.dist import bind_to_gpu_numa
        numa_cpus = bind_to_gpu_numa(local)   # before any pinned allocation
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        # stdout carries the one JSON line only: NCCL's banner ("NCCL version ...", printed to stdout when the
        # communicator is created) goes to stderr
        sys.stdout.flush()
        keep = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=dev)
            dist.barrier()
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(keep, 1)
            os.close(keep)
    E, N, ROT = args.envs, N_AGENTS, args.rot
    K = args.steps
    NW = min(args.windows, K)
    sampler = ClockSampler(local) if rank == 0 else None   # started early: it is warm when the timed region begins
    T = Timer(torch, dist, dev, world)
    main_stream = T.main

    extra = {"max_touching": args.max_touching} if args.max_touching else {}
    sims = [gym_macm.BatchedFlock(E, n_agents=[N], reward_mode="linear", device=dev, seed=1234 + 1000 * rank + r, **extra)
            for r in range(ROT)]
    # U{0,1,2}^3 per agent-step, pre-generated on the device (a pool cycled through)
    g = torch.Generator(device=dev)
    g.manual_seed(99 + rank)
    POOL = 61   # prime: batch r at its j-th step uses action set (j + 7 r) mod POOL, all distinct in sequence
    acts = torch.zeros((POOL, E, N, 4), dtype=torch.uint8, device=dev)
    acts[..., :3] = torch.randint(0, 3, (POOL, E, N, 3), generator=g, device=dev, dtype=torch.uint8)

    NS = max(1, min(args.streams, ROT))
    # gym_macm.BatchPool (the public API for this): the rotation's batches round-robin over NS streams of their own
    pool = gym_macm.BatchPool(sims, n_streams=NS) if NS > 1 else None
    streams = pool.streams if pool else []
    if pool is None:
        for s_ in sims:
            s_.engine.stream = None

    def act_of(k):
        return acts[(k // ROT + 7 * (k % ROT)) % POOL]

    def step_on(strs):
        def issue(k):
            s = sims[k % ROT]
            st = strs[(k % ROT) % len(strs)] if strs else main_stream
            if args.policy == "flock":
                with torch.cuda.stream(st):
                    a = s.bot_actions("flock")
            else:
                a = act_of(k)
            s.engine.step(a, st)
        return issue

    def pool_issue(k):           # the headline path: BatchPool.step
        if args.policy == "flock":
            s = sims[k % ROT]
            with torch.cuda.stream(s.engine.stream):
                a = s.bot_actions("flock")
        else:
            a = act_of(k)
        pool.step(a)

    # settle: every batch runs SETTLE steps (1.07 s of simulated time of a 60 s / 3601-step episode)
    # so that the overlaps of the random spawn are resolved; then W warm-up steps of the rotation
    issue, issue1 = (pool_issue if pool else step_on([])), step_on([])
    if pool:
        pool.k = 0
    for k in range(args.settle * ROT):
        issue1(k)
    torch.cuda.synchronize()
    for st in streams:
        st.wait_stream(main_stream)
    for k in range(args.warmup):
        issue(k)
    torch.cuda.synchronize()
    if pool:
        pool.k = 0
    launches0 = sum(s.engine.launch_count for s in sims)
    t0 = time.time()
    ms_per_step, ms_all, knext = T.windows(issue, K, NW, streams)
    t1 = time.time()
    launches = sum(s.engine.launch_count for s in sims) - launches0
    clocks = sampler.stop(t0, t1) if sampler else None
    torch.cuda.synchronize()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, sims[(K - 1) % ROT])   # the batch the last timed step stepped
    for s_ in sims:                  # the legs below name their streams themselves
        s_.engine.stream = None
    value = world * E * N / (ms_per_step * 1e-3)

    legs = {}
    plain = args.policy == "random" and not args.no_legs
    # ---- further device-timed legs on the same batches ------------------------------------------------------
    # (1) everything on ONE stream: every launch waits for the last env of the one before it (the r1 headline)
    if plain and NS > 1:
        T.windows(issue1, min(K, 200), 1)     # warm-up of this shape
        ms1, all1, _ = T.windows(issue1, K, NW)
        legs["one_stream"] = {"value": world * E * N / (ms1 * 1e-3), "unit": UNIT, "ms_per_step": ms1,
                               "windows": NW, "note": "the same steps on one stream: no overlap between a batch's "
                               "tail (a few envs with long contact islands) and the next batch"}
    # (2) one launch alone on an idle GPU (synchronised on both sides): the kernel's own duration, read from the
    #     kernel's trace hook (macm_set_trace: every warp records %globaltimer at entry and exit; duration = last
    #     exit - first entry, so no launch or event latency is in it)
    iso = None
    if plain:
        import ctypes as C
        from gym_macm import _lib
        trace = torch.zeros((E, 4), dtype=torch.int64, device=dev)
        durs = []
        for k in range(24):
            s_ = sims[k % ROT]
            _lib.check(_lib.lib().macm_set_trace(s_.engine._h, C.c_void_p(trace.data_ptr())))
            torch.cuda.synchronize()
            s_.engine.step(act_of(knext + k))
            torch.cuda.synchronize()
            _lib.check(_lib.lib().macm_set_trace(s_.engine._h, None))
            durs.append(float(trace[:, 1].max() - trace[:, 0].min()) * 1e-6)   # ns -> ms
        iso = T.max_over_ranks(statistics.median(durs[4:]))
        del trace
    # (3) macm_rollout: R steps of a batch per launch, the envs' bodies held on chip between the steps; every
    #     step still writes its obs / nn_idx / rewards / collided / done (to per-step arrays).
    if plain and args.rollout > 0:
        R = min(args.rollout, POOL)
        outs = [sims[0].engine.rollout_buffers(R) for _ in range(2)]
        n_launch = max(ROT, (min(K, 2000) // R) // ROT * ROT)

        def roll(j):
            sims[j % ROT].engine.rollout(acts[:R], R, None, 0, outs[j & 1])
        T.windows(roll, ROT, 1)
        msr, _, _ = T.windows(roll, n_launch, 1)      # ms per launch of R steps
        legs["rollout"] = {"value": world * E * N * R / (msr * 1e-3), "unit": UNIT,
                            "ms_per_step": msr / R, "steps_per_launch": R, "launches": n_launch,
                            "note": "macm_rollout, per-step outputs written every step; bit-identical to single steps "
                                    "(tests/test_gpu_rollout.py)"}
        del outs

    # live contacts per agent (c-bar of the roofline formula), measured on this rank's batches
    c_bar = float(sum(float(s.state["contact_count"].sum()) for s in sims) / (ROT * E * N))
    touching = float(sum(float(s.state["env_state"][:, 2].sum()) for s in sims) / (ROT * E))
    overflow = [sum(x) for x in zip(*[s.overflow_count() for s in sims])]
    b_alg = b_alg_per_agent_step(c_bar, 1, N)
    peak, peak_kind = measured_peak()
    achieved = b_alg * E * N / (ms_per_step * 1e-3) / 1e9   # GB/s of ONE GPU's kernel
    static = {}
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            static = json.load(f)
    except Exception:
        pass

    # ---- the exchange BASELINE config 5 names: obs + rewards (+ done) of every shard to a learner rank ------
    if world > 1 and plain:
        from gym_macm.dist import PeerGather
        nbytes_in = (world - 1) * E * N * (16 + 4) + (world - 1) * E   # into the learner per step
        # (a) the step kernel stores its outputs into rank 0's buffers itself (NVLink peer stores, no collective)
        peer = PeerGather(sims[0], world * E, learner=0, names=("obs", "rewards", "done"))

        def peer_step(k):
            s = sims[k % ROT]
            st = streams[(k % ROT) % NS] if streams else None
            s.engine.rollout(act_of(k), 1, None, 0, peer.mine[k & 1], st)
        T.windows(peer_step, min(K, 100), 1, streams)
        msp, _, _ = T.windows(peer_step, K, NW, streams)
        legs["gather_peer"] = {"value": world * E * N / (msp * 1e-3), "unit": UNIT, "ms_per_step": msp,
                                "bytes_into_learner_per_step": nbytes_in,
                                "learner_ingress_GBps": nbytes_in / (msp * 1e-3) / 1e9, "windows": NW,
                                "note": "obs+rewards+done of every rank stored into rank 0's buffers by the step kernel "
                                        "itself (gym_macm.dist.PeerGather: NVLink peer stores through CUDA IPC, no collective)"}
        # (b) NCCL all-gather of obs + rewards on a side stream: the next batch steps while this one's outputs travel
        gathered = [torch.empty((world,) + tuple(sims[0].state[k_].shape), dtype=sims[0].state[k_].dtype, device=dev)
                    for k_ in ("obs", "rewards")]
        gstream = torch.cuda.Stream(device=dev)

        def nccl_step(k):
            s = sims[k % ROT]
            s.engine.step(act_of(k))
            gstream.wait_stream(main_stream)
            with torch.cuda.stream(gstream):
                dist.all_gather_into_tensor(gathered[0], s.state["obs"])
                dist.all_gather_into_tensor(gathered[1], s.state["rewards"])

        def join():
            main_stream.wait_stream(gstream)
        T.windows(nccl_step, min(K, 50), 1, after=join)
        msn, _, _ = T.windows(nccl_step, K, NW, after=join)
        legs["gather_nccl"] = {"value": world * E * N / (msn * 1e-3), "unit": UNIT, "ms_per_step": msn,
                                "bytes_into_every_rank_per_step": (world - 1) * E * N * 20,
                                "ingress_GBps": (world - 1) * E * N * 20 / (msn * 1e-3) / 1e9,
                                "note": "NCCL all_gather_into_tensor of obs and rewards to every rank, on a side stream"}
        peer.close()
        del gathered, peer

    # ---- the other BASELINE configs, each rotated over more than 2x L2 ----------------------------------------
    if plain:
        legs["configs"] = other_configs(torch, gym_macm, T, dev, world, rank, K, NW, peak, args.settle)

    # ---- end to end through the host-buffer entry point (macm_step_host) --------------------
    # DEPTH batches in rotation (the usual double/triple-buffered rollout): while one batch's
    # observations travel to the host, the others step.  Every step still pays its own H2D of actions
    # (from pinned host memory, where the host policy left them) and its own D2H of obs + rewards +
    # done inside the timed region, and the host reads a result before it issues the batch's next step.
    DEPTH = max(1, min(args.e2e_depth, ROT))
    pp = sims[:DEPTH] if args.e2e_steps > 0 else []
    # Two result sets, both contiguous in the output slab (ONE device->host transfer each):
    #   e2e      obs floats + rewards + done: what a learner consumes (the definition of round 1's line)
    #   e2e_all  + nearest-agent ids + collided flags: everything the drop-in Flock.step marshals into its dicts
    #            (mvmnt.py:140,163-178,204-220)
    pin = pp[0].engine.pinned() if pp else {}
    host_actions = [acts[i].cpu().pin_memory() for i in range(4)]

    def e2e_leg(want, steps):
        for s_ in pp:
            for k in range(3):
                s_.engine.step_host(host_actions[k % 4], want=want)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        checksum = 0.0
        te = time.perf_counter()
        for k in range(steps):
            cur = pp[k % DEPTH].engine
            if k >= DEPTH:
                cur.host_sync()                                   # results of this batch's previous step
                checksum += float(cur.pinned()["rewards"][0, 0])  # the host reads them
            cur.step_host(host_actions[k % 4], want=want, wait=False)
        for s_ in pp:
            s_.engine.host_sync()
        el = T.max_over_ranks(time.perf_counter() - te)
        h2d = int(host_actions[0].numel() * host_actions[0].element_size())
        d2h = int(sum(pin[k].numel() * pin[k].element_size() for k in want))
        return {"value": world * E * N * steps / el, "unit": UNIT, "h2d_bytes_per_step": h2d,
                "d2h_bytes_per_step": d2h, "steps": steps, "d2h_transfers_per_step": 1,
                "pcie_GBps_per_gpu": (h2d + d2h) * steps / el / 1e9, "outputs": list(want)}

    e2e = None
    if pp:
        e2e = e2e_leg(("obs", "rewards", "done"), args.e2e_steps)
        e2e["path"] = ("macm_step_host_async/macm_host_sync on %d batches in rotation: pinned host actions -> device, step "
                       "kernel, obs + rewards + done -> pinned host in ONE transfer (output slab)" % DEPTH)
        if plain:
            legs["e2e_all"] = e2e_leg(("obs", "rewards", "done", "nn_idx", "collided"), max(60, args.e2e_steps // 2))
            legs["e2e_all"]["note"] = "every output of the drop-in Flock.step (obs floats, nearest-agent ids, rewards, collided, done)"

    if rank == 0:
        cpu = None
        if world == 1:
            try:
                from oracle import oracle
                oracle.build()
                cores = len(os.sched_getaffinity(0))
                n_envs = min(N_ENVS, cores * 64)   # 64 envs per thread and step: thread start/join well amortised
                rate, st, el = cpu_oracle_rate(n_envs, cores, args.cpu_seconds)
                rate1, st1, el1 = cpu_oracle_rate(8, 1, min(3.0, args.cpu_seconds))   # single process, one thread
                cpu = {"value": rate, "unit": UNIT, "cores": cores, "kind": "port",
                       "sample": "%d envs x %d agents x %d steps in %.1f s; CPU restatement (oracle/), not pybox2d"
                                 % (n_envs, N, st, el),
                       "single_thread": {"value": rate1, "unit": UNIT, "cores": 1,
                                         "sample": "8 envs x %d agents x %d steps in %.1f s" % (N, st1, el1)}}
                probe = pybox2d_probe(seconds=3.0)
                cpu["pybox2d_probe"] = probe
                real = probe.get("reference_loop") if probe.get("available") else None
                if real and "agent_steps_per_sec" in real:
                    cpu["pybox2d"] = {"value": real["agent_steps_per_sec"], "unit": UNIT, "cores": 1, "kind": "pybox2d",
                                      "sample": "the reference's Flock.step loop, %d steps in %.1f s" % (real["steps"], real["seconds"])}
            except Exception as ex:  # the checker missing must not hide the GPU number
                cpu = {"value": None, "unit": UNIT, "cores": 0, "kind": "port", "sample": "failed: %r" % (ex,)}
        info = sims[0].engine.info
        kname = "macm_step_kernel<%d,%d,0,0>" % (info.lanes_per_env, info.agents_per_lane)
        roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                    "traffic": static.get("dram_bytes_per_launch"),
                    "traffic_kind": "static: %s" % static.get("source", "profiles/traffic.json"),
                    "peak_kind": peak_kind, "bytes_per_agent_step": b_alg, "kernel": kname,
                    "kernel_ms": ms_per_step,
                    "kernel_ms_kind": "launch-to-launch interval of the timed region (consecutive launches overlap: "
                                      "programmatic dependent launch, %d streams)" % NS}
        if iso:
            roofline["kernel_ms_isolated"] = iso
            roofline["kernel_ms_isolated_kind"] = ("first warp entry to last warp exit (%globaltimer, macm_set_trace) of a "
                                                    "launch alone on an idle, synchronised GPU; median of 20")
            roofline["frac_isolated"] = b_alg * E * N / (iso * 1e-3) / 1e9 / peak
        # what actually bounds the kernel (profiles/README.md): warp-instruction issue.  The instruction count is
        # the ncu figure of the committed capture; the peak is one instruction per clock on each of the SMs' four
        # sub-partitions.
        inst = static.get("warp_inst_per_env_step")
        roofline_issue = None
        if inst:
            sm_clock = (clocks or {}).get("sm_mhz") or 1965.0
            nsp = info.sm_count * 4
            floor_ms = inst * E / (nsp * sm_clock * 1e6) * 1e3
            roofline_issue = {"bound": "issue", "warp_inst_per_env_step": inst, "inst_kind": "static: %s" % static.get("source"),
                              "sub_partitions": nsp, "sm_mhz": sm_clock, "floor_ms": floor_ms,
                              "achieved": inst * E / (ms_per_step * 1e-3) / 1e12, "peak": nsp * sm_clock * 1e6 / 1e12,
                              "unit": "T warp-inst/s", "frac": floor_ms / ms_per_step}
        out = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K,
            "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "windows": NW, "window_ms": ms_all,
            "window_agg": "%d steps in %d window(s) between barrier+synchronize; per-rank median of the time per step "
                          "over the windows, max over ranks" % (K, NW),
            "config": {"workload": WORKLOAD, "envs_per_gpu": E, "agents_per_env": N, "reward_mode": "linear",
                       "actions": "pre-generated on device, U{0,1,2}^3" if args.policy == "random" else "bots.flock on device",
                       "l2": "inputs larger than L2: rotation over %d independent batches (%.0f MB of state+outputs)"
                             % (ROT, ROT * E * N * 73 / 1e6),
                       "streams": NS, "numa_bound_cpus": len(numa_cpus) if numa_cpus else None,
                       "damping_model": default_damping(),
                       "parallelism": "envs sharded, %d per GPU, no data-path collective" % E,
                       "launch": {"lanes_per_env": info.lanes_per_env, "agents_per_lane": info.agents_per_lane,
                                  "threads_per_block": info.threads_per_block, "blocks": info.blocks,
                                  "smem_per_block": info.smem_bytes_per_block, "blocks_per_sm": info.blocks_per_sm},
                       "settle_steps_per_batch": args.settle,
                       "contacts_per_agent": c_bar, "touching_contacts_per_env": touching,
                       "envs_with_contact_overflow": overflow},
            "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches),
            "roofline": roofline, "roofline_issue": roofline_issue,
            "cpu_baseline": cpu,
        }
        out.update(legs)
        print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


def other_configs(torch, gym_macm, T, dev, world, rank, K, NW, peak, settle):
    """BASELINE configs 3, 4 and the 16M-agent point of config 5: device-timed like the headline (independent
    batches alternating between two streams, footprint of the rotation > 2x the 126 MB L2), each with its own
    algorithmic bytes per agent-step (SURVEY 8d) and roofline fraction."""
    out = {}
    g = torch.Generator(device=dev)
    g.manual_seed(7 + rank)
    st2 = [torch.cuda.Stream(device=dev) for _ in range(2)]

    def run(name, sims, acts, n_agents, b_alg_fn, steps, workload):
        ROT, POOL = len(sims), acts.shape[0]
        E = sims[0].engine.E

        def issue(k):
            sims[k % ROT].engine.step(acts[(k // ROT + 7 * (k % ROT)) % POOL], st2[(k % ROT) & 1])
        for k in range(settle * ROT):
            sims[k % ROT].engine.step(acts[(k // ROT + 7 * (k % ROT)) % POOL])
        torch.cuda.synchronize()
        T.windows(issue, min(steps, 4 * ROT), 1, st2)
        per, win_ms, _ = T.windows(issue, steps, NW, st2)
        c_bar = float(sum(float(s.state["contact_count"].sum()) for s in sims) / (ROT * E * n_agents))
        b = b_alg_fn(c_bar)
        ach = b * E * n_agents / (per * 1e-3) / 1e9
        foot = sum(sum(t.numel() * t.element_size() for t in s.state.values()) for s in sims)
        ov = [sum(x) for x in zip(*[s.overflow_count() for s in sims])]
        out[name] = {"workload": workload, "value": world * E * n_agents / (per * 1e-3), "unit": UNIT,
                     "ms_per_step": per, "steps": steps, "windows": len(win_ms), "envs_per_gpu": E, "agents_per_env": n_agents,
                     "batches_in_rotation": ROT, "footprint_MB": foot / 1e6, "contacts_per_agent": c_bar,
                     "bytes_per_agent_step": b, "envs_with_contact_overflow": ov,
                     "roofline": {"bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak}}

    # config 3: multi-flock, 6 agents, targets=[0,0,1,1,2,2], 65,536 envs, binary reward
    E3, N3 = 65536, 6
    sims = [gym_macm.BatchedFlock(E3, n_agents=[N3], targets=[0, 0, 1, 1, 2, 2], device=dev, seed=31 + 100 * rank + r)
            for r in range(10)]
    acts = torch.zeros((31, E3, N3, 4), dtype=torch.uint8, device=dev)   # a prime pool: no short action cycle
    acts[..., :3] = torch.randint(0, 3, (31, E3, N3, 3), generator=g, device=dev, dtype=torch.uint8)
    run("config3_multi_flock", sims, acts, N3, lambda c: b_alg_per_agent_step(c, 3, N3), K,
        "cm-flock-v0 6 agents, targets=[0,0,1,1,2,2], x 65536 envs per GPU, binary reward")
    del sims, acts
    # config 4: team deathmatch, 3 teams x 15 agents, 16,384 envs
    E4, N4 = 16384, 45
    sims = [gym_macm.BatchedTDM(E4, n_agents=[15, 15, 15], device=dev, seed=41 + 100 * rank + r) for r in range(2)]
    acts = torch.randint(0, 3, (17, E4, N4, 4), generator=g, device=dev, dtype=torch.uint8)
    acts[..., 3] = torch.randint(0, 2, (17, E4, N4), generator=g, device=dev, dtype=torch.uint8)
    run("config4_tdm", sims, acts, N4, lambda c: 828.0 + 32.0 * c, max(4, min(K, 100)),
        "cm-tdm-v0 3 teams x 15 agents x 16384 envs per GPU, random actions with attacks")
    del sims, acts
    # config 5: 64-agent flock envs, 32,768 per GPU (16.8M agents on 8 GPUs), no exchange here (see gather_* legs)
    E5, N5 = 32768, N_AGENTS
    sims = [gym_macm.BatchedFlock(E5, n_agents=[N5], reward_mode="linear", device=dev, seed=51 + 100 * rank + r)
            for r in range(2)]
    acts = torch.zeros((31, E5, N5, 4), dtype=torch.uint8, device=dev)
    acts[..., :3] = torch.randint(0, 3, (31, E5, N5, 3), generator=g, device=dev, dtype=torch.uint8)
    run("config5_32768_envs_per_gpu", sims, acts, N5, lambda c: b_alg_per_agent_step(c, 1, N5), max(4, min(K, 100)),
        "cm-flock-v0 64 agents x 32768 envs per GPU (%.1fM agents on %d GPUs), linear reward" % (world * E5 * N5 / 1e6, world))
    if world > 1:
        import torch.distributed as dist
        from gym_macm.dist import PeerGather
        steps = max(4, min(K, 40))
        peer = PeerGather(sims[0], world * E5, learner=0, names=("obs", "rewards", "done"))

        def peer_step(k):
            sims[k % 2].engine.rollout(acts[(k // 2 + 7 * (k % 2)) % 31], 1, None, 0, peer.mine[k & 1], st2[k & 1])
        T.windows(peer_step, 4, 1, st2)
        msp, _, _ = T.windows(peer_step, steps, NW, st2)
        nb = (world - 1) * (E5 * N5 * 20 + E5)
        out["config5_32768_envs_per_gpu"]["gather_peer"] = {
            "value": world * E5 * N5 / (msp * 1e-3), "unit": UNIT, "ms_per_step": msp,
            "bytes_into_learner_per_step": nb, "learner_ingress_GBps": nb / (msp * 1e-3) / 1e9}
        gathered = [torch.empty((world,) + tuple(sims[0].state[k_].shape), dtype=sims[0].state[k_].dtype, device=dev)
                    for k_ in ("obs", "rewards")]
        gstream = torch.cuda.Stream(device=dev)

        def nccl_step(k):
            s = sims[k % 2]
            s.engine.step(acts[(k // 2 + 7 * (k % 2)) % 31])
            gstream.wait_stream(T.main)
            with torch.cuda.stream(gstream):
                dist.all_gather_into_tensor(gathered[0], s.state["obs"])
                dist.all_gather_into_tensor(gathered[1], s.state["rewards"])

        def join():
            T.main.wait_stream(gstream)
        T.windows(nccl_step, 4, 1, after=join)
        msn, _, _ = T.windows(nccl_step, steps, NW, after=join)
        out["config5_32768_envs_per_gpu"]["gather_nccl"] = {
            "value": world * E5 * N5 / (msn * 1e-3), "unit": UNIT, "ms_per_step": msn,
            "bytes_into_every_rank_per_step": (world - 1) * E5 * N5 * 20,
            "ingress_GBps": (world - 1) * E5 * N5 * 20 / (msn * 1e-3) / 1e9}
        peer.close()
        del gathered, peer
    return out


if __name__ == "__main__":
    main()
