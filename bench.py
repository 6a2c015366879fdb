#!/usr/bin/env python
"""bench.py -- headline benchmark of the B200-native ReVolt dynamic-positioning hot path.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--envs-per-gpu E] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W

Workload (BASELINE.json configs[2], SURVEY.md section 8d config 3): RevoltFinal(extended_state, cont_ang)
env step -- action transform, 20 sub-steps of the 3-DOF stand-in hull, body-frame error, observation, reward,
termination, 400-step episodes with in-kernel re-sampling -- on 16 Mi environments PER GPU (weak scaling;
environments shard by global index, no data-path collective), fresh U(-1,1)^7 actions every step.
A "step" is one pass of the hot path over the whole batch = exactly one env_step_kernel launch per GPU.

One JSON line on stdout (rank 0):
  value      env-steps/s over all GPUs, inputs resident in HBM, CUDA-event timed, max over ranks
  e2e        same metric through the public API (ml4ca_b200.env.RevoltFinal.step -> C ABI) with HOST buffers:
             every step copies that step's actions from pinned host memory and reads obs/reward/done back
  roofline   HBM roofline of the env-step kernel: 177 algorithmic bytes per env-step (SURVEY.md 8d)
  cpu_baseline  the CPU oracle (vectorised NumPy port of the reference wrapper + float64 hull) on a bounded sample
  extra      secondary kernels of the path (QP allocations/s, pseudoinverse+PID/s, ...), each with its own roofline

--dump-outputs DIR writes what the last timed step returned to its caller (rank 0) as DIR/<name>.npy, so that two builds
run with the same arguments -- hence the same seeded inputs -- can be compared output for output.
"""
import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
# stdout carries exactly one JSON line.  NCCL writes its version / debug banner to file descriptor 1 from C (at WARN level
# too), so descriptor 1 is pointed at stderr for the whole run and the JSON line goes to a duplicate of the real stdout.
# NCCL_DEBUG is left exactly as the caller set it (the driver reads the rank count out of an INFO log).
_REAL_STDOUT = os.fdopen(os.dup(1), "w")
sys.stdout.flush()
os.dup2(2, 1)


def emit(line):
    _REAL_STDOUT.write(json.dumps(line) + "\n")
    _REAL_STDOUT.flush()


ENV_STEP_BYTES = 177      # SURVEY.md 8(d): read 60 state + 28 action, write 48 state + 36 obs + 4 rew + 1 done
ENV_STEP_TRAFFIC = 2.9137e9  # measured DRAM bytes of one 16 Mi-env launch (profiles/env_step_r1.md, capture prof_env_r1h); algorithmic: 2.9696e9
PINV_PID_BYTES = 80       # read eta, nu, ref, integ (48) + write integ, n, alpha (32)
QP_BYTES = 68             # read tau 3 + prev 5 words, write x 8 + status 1
POLICY_BYTES = 72         # read obs 36, write action 28 + value 4 + logp 4
ROLLOUT_TRAIN_BYTES = 185  # state r/w 108 + trajectory record 77 (SURVEY.md 8d)
GAE_BYTES = 17            # read r, V, flag byte; write A, R
ACTION_POOL = 2           # flat U(-1,1) buffers; step i reads a [7, n] window at a new offset: fresh actions per (env, step)
ACTION_SHIFT = 4 * 1031   # floats between consecutive windows (16-byte aligned, so the vectorised kernel path is kept)
DUMP_ENVS = 1 << 19       # environments sampled by --dump-outputs: 11 float32 outputs + 1 float64 index each, 27 MB in all


def load_tensor_peak():
    """Sustained dense bf16/fp16 TFLOP/s (MEASURED_PEAKS.json), else the profiling guide's nominal figure."""
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as fh:
            p = json.load(fh)
        if "bf16_tflops_sustained" in p:
            return float(p["bf16_tflops_sustained"]), "measured sustained (MEASURED_PEAKS.json)"
    return 2250.0, "nominal dense bf16 (B200_PROFILING.md)"


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as fh:
            p = json.load(fh)
        return float(p["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler(threading.Thread):
    """Polls NVML for SM clock and throttle reasons while the timed region runs."""

    REASONS = {0x1: "gpu_idle", 0x2: "applications_clocks_setting", 0x4: "sw_power_cap", 0x8: "hw_slowdown",
               0x10: "sync_boost", 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown",
               0x80: "hw_power_brake_slowdown", 0x100: "display_clock_setting"}

    def __init__(self, index, period=0.004):
        super().__init__(daemon=True)
        self.index, self.period = index, period
        self.samples, self.marks = [], {}
        self.stop_flag = threading.Event()
        self.ok = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception as e:  # noqa: BLE001
            self.err = repr(e)

    def run(self):
        if not self.ok:
            return
        while not self.stop_flag.is_set():
            try:
                mhz = self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM)
                try:
                    rs = self.nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:  # noqa: BLE001
                    rs = self.nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                self.samples.append((time.perf_counter(), mhz, rs))
            except Exception:  # noqa: BLE001
                pass
            time.sleep(self.period)

    def mark(self, name):
        self.marks[name] = time.perf_counter()

    def summary(self):
        if not self.ok or not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvml_unavailable"]}
        t0, t1 = self.marks.get("start", 0), self.marks.get("end", float("inf"))
        inside = [s for s in self.samples if t0 <= s[0] <= t1] or self.samples
        mhz = sorted(s[1] for s in inside)
        bits = 0
        for s in inside:
            bits |= s[2]
        reasons = [n for b, n in self.REASONS.items() if bits & b and n != "gpu_idle"]
        return {"sm_mhz": mhz[len(mhz) // 2], "sm_max_mhz": self.max_mhz, "reasons": reasons, "samples": len(inside)}


# ---- CPU side (oracle port) --------------------------------------------------------------------------------------
def _cpu_worker(args):
    n, steps, seed = args
    import numpy as np
    from oracle import env_oracle as EO
    spec = EO.EnvSpec('final', True, True, max_ep_len=800)
    rng = np.random.default_rng(seed)
    st = EO.new_state(spec, n)
    EO.reset(spec, st, seed=seed, fraction=0.8)
    acts = rng.uniform(-1, 1, (steps, 7, n))
    t0 = time.perf_counter()
    for t in range(steps):
        o, r, d, info = EO.step(spec, st, acts[t])
        ended = d | info['truncated']
        if ended.any():
            EO.reset(spec, st, mask=ended, seed=seed, fraction=0.8)
    return time.perf_counter() - t0


def cpu_env_steps_per_s(n_total=1 << 16, steps=8, cores=None):
    """The CPU oracle (vectorised NumPy port of customEnv.py + float64 hull) on `cores` processes."""
    import multiprocessing as mp
    cores = cores or os.cpu_count() or 1
    per = max(1, n_total // cores)
    ctx = mp.get_context("fork")
    with ctx.Pool(cores) as pool:
        busy = pool.map(_cpu_worker, [(per, steps, 1000 + i) for i in range(cores)])
    wall = max(busy)               # slowest worker's stepping loop (process start-up and imports excluded)
    return per * cores * steps / wall, cores, "%d envs x %d steps (RevoltFinal ext+cont, float64 NumPy port, %d processes)" % (
        per * cores, steps, cores)


def _cpu_qp_worker(args):
    lo, hi = args
    from ml4ca_b200 import synth
    from oracle import qp_oracle as QO
    tau, prev = synth.qp_batch(4096, seed=0)
    t0 = time.perf_counter()
    for j in range(lo, hi):
        QO.solve_stock(tau[:, j], prev[:, j])
    return time.perf_counter() - t0


def cpu_qp_allocations_per_s(n_solves=512, cores=None):
    """The reference NLP on SciPy SLSQP (oracle restatement of QPTA.solve_QP, bit-identical to the reference code in the
    build container) on the first n_solves demands of the config-1 batch, split over `cores` processes."""
    import multiprocessing as mp
    cores = cores or os.cpu_count() or 1
    per = max(1, n_solves // cores)
    ctx = mp.get_context("fork")
    use_ref = reference_code_available()
    with ctx.Pool(cores) as pool:
        busy = pool.map(_refcode_qp_worker if use_ref else _cpu_qp_worker, [(i * per, (i + 1) * per) for i in range(cores)])
    wall = max(busy)          # slowest worker's solve loop (process start-up and imports excluded)
    return {"value": per * cores / wall, "unit": "allocations/s", "cores": cores, "kind": "reference" if use_ref else "port",
            "single_core_ms_per_solve": 1e3 * sum(busy) / (per * cores),
            "sample": "first %d demands of the 4096-sample config-1 batch, %s on SciPy SLSQP (reference defaults), %d processes"
                      % (per * cores, "the reference's QPTA.solve_QP" if use_ref else "oracle restatement of QPTA.solve_QP", cores)}


def reference_code_available():
    from oracle import ref_loader
    return ref_loader.available()


def _refcode_env_worker(args):
    """The REFERENCE CODE: customEnv.RevoltFinal objects (imported unmodified from /root/reference or from the byte-compiled
    oracle/_ref) stepped one env at a time, as the reference does, on the float64 stand-in twin."""
    n_envs, steps, seed = args
    import numpy as np
    from oracle import ref_loader, vessel
    mod = ref_loader.load_env_module()
    np.random.seed(seed)
    envs = [mod.RevoltFinal(vessel.VesselTwin(), cont_ang=True, extended_state=True) for _ in range(n_envs)]
    for e in envs:
        e.reset(fraction=0.8)
    rng = np.random.default_rng(seed)
    acts = rng.uniform(-1, 1, (steps, n_envs, 7))
    t0 = time.perf_counter()
    for t in range(steps):
        for k, e in enumerate(envs):
            o, r, d, _ = e.step(acts[t, k])
            if d:
                e.reset(fraction=0.8)
    return time.perf_counter() - t0


def refcode_env_steps_per_s(envs_per_core=8, steps=100, cores=None):
    import multiprocessing as mp
    from oracle import ref_loader
    cores = cores or os.cpu_count() or 1
    with mp.get_context("fork").Pool(cores) as pool:
        busy = pool.map(_refcode_env_worker, [(envs_per_core, steps, 7000 + i) for i in range(cores)])
    wall = max(busy)
    return envs_per_core * cores * steps / wall, cores, (
        "%d reference RevoltFinal objects (%s) x %d steps on the float64 stand-in twin, %d processes"
        % (envs_per_core * cores, ref_loader.source(), steps, cores))


def _refcode_qp_worker(args):
    lo, hi = args
    import numpy as np
    from ml4ca_b200 import synth
    from oracle import ref_loader
    qp = ref_loader.load_qp_module()
    ta = qp.QPTA()
    tau, prev = synth.qp_batch(4096, seed=0)
    t0 = time.perf_counter()
    for j in range(lo, hi):
        ta.previous_thruster_state = [float(v) for v in prev[:, j]] + [np.pi / 2]
        ta.solve_QP(tau[:, j].reshape(3, 1))
    return time.perf_counter() - t0


_REF_STATE = {}


def _ref_init(per, seed_base):
    """Pool initializer: every worker process builds its own batch of oracle envs once and keeps it between steps."""
    import numpy as np
    from oracle import env_oracle as EO
    seed = seed_base + os.getpid() % 100000
    spec = EO.EnvSpec('final', True, True, max_ep_len=800)
    st = EO.new_state(spec, per)
    EO.reset(spec, st, seed=seed, fraction=0.8)
    _REF_STATE.update(spec=spec, st=st, rng=np.random.default_rng(seed), seed=seed, EO=EO, per=per)


def _ref_step(inner):
    S = _REF_STATE
    EO, spec, st = S["EO"], S["spec"], S["st"]
    acts = S["rng"].uniform(-1, 1, (inner, 7, S["per"]))
    t0 = time.perf_counter()
    for t in range(inner):
        o, r, d, info = EO.step(spec, st, acts[t])
        ended = d | info['truncated']
        if ended.any():
            EO.reset(spec, st, mask=ended, seed=S["seed"], fraction=0.8)
    return time.perf_counter() - t0


def run_reference(args, rank, world):
    """--impl reference: the reference's own CPU implementation of the path, timed on the host cores.
    The reference is Python and cannot travel to the GPU box, so this is the oracle port (kind 'port'): the vectorised
    NumPy restatement of customEnv.py + the float64 hull, one persistent process per core (the env batches live in the
    workers across steps, so a bench step times stepping only).  One bench step = `inner` env steps of 64 Ki envs."""
    if rank != 0:
        return
    if reference_code_available() and not os.environ.get("ML4CA_REFERENCE_PORT"):
        return run_reference_code(args, world)
    import multiprocessing as mp
    cores = os.cpu_count() or 1
    n_total, inner = 1 << 16, 8
    per = max(1, n_total // cores)
    ctx = mp.get_context("fork")

    def serve(conn, idx):                       # one dedicated process per core: exactly one task per core and step
        _ref_init(per, 4000 + idx)
        while True:
            k = conn.recv()
            if k <= 0:
                break
            conn.send(_ref_step(k))

    pipes, procs = [], []
    for c in range(cores):
        a, b = ctx.Pipe()
        pr = ctx.Process(target=serve, args=(b, c), daemon=True)
        pr.start()
        pipes.append(a), procs.append(pr)

    def step_all(k):
        for a in pipes:
            a.send(k)
        return [a.recv() for a in pipes]

    for _ in range(max(1, min(args.warmup, 2))):
        step_all(1)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step_all(inner)
    wall = time.perf_counter() - t0
    for a in pipes:
        a.send(0)
    for pr in procs:
        pr.join(timeout=5)
    n_total = per * cores
    value = n_total * inner * args.steps / wall
    sample = "%d envs x %d env-steps per bench step, %d bench steps, %d persistent processes" % (n_total, inner, args.steps, cores)
    line = {
        "impl": "reference", "metric": "env_steps_per_sec", "value": value, "unit": "env-steps/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * wall / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(args, world),
        "cpu_baseline": {"value": value, "unit": "env-steps/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


def run_reference_code(args, world):
    """--impl reference with the reference's own code on the box (oracle/_ref or the checkout): customEnv.RevoltFinal
    objects stepped one by one, as ppo.py:293 does, one persistent process per core.  kind = "reference".  The vectorised
    NumPy port (what --impl reference timed in round 1; ML4CA_REFERENCE_PORT=1 still selects it) is ~300x faster per core
    than the reference code and is reported next to it."""
    import multiprocessing as mp
    from oracle import ref_loader
    cores = os.cpu_count() or 1
    per, inner = 8, 25
    ctx = mp.get_context("fork")

    def serve(conn, idx):
        import numpy as np
        from oracle import vessel
        mod = ref_loader.load_env_module()
        np.random.seed(9000 + idx)
        envs = [mod.RevoltFinal(vessel.VesselTwin(), cont_ang=True, extended_state=True) for _ in range(per)]
        for e in envs:
            e.reset(fraction=0.8)
        rng = np.random.default_rng(9000 + idx)
        while True:
            k = conn.recv()
            if k <= 0:
                break
            acts = rng.uniform(-1, 1, (k, per, 7))
            t0 = time.perf_counter()
            for t in range(k):
                for j, e in enumerate(envs):
                    o, r, d, _ = e.step(acts[t, j])
                    if d:
                        e.reset(fraction=0.8)
            conn.send(time.perf_counter() - t0)

    pipes, procs = [], []
    for c in range(cores):
        a, b = ctx.Pipe()
        pr = ctx.Process(target=serve, args=(b, c), daemon=True)
        pr.start()
        pipes.append(a), procs.append(pr)

    def step_all(k):
        for a in pipes:
            a.send(k)
        return [a.recv() for a in pipes]

    for _ in range(max(1, min(args.warmup, 2))):
        step_all(2)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step_all(inner)
    wall = time.perf_counter() - t0
    for a in pipes:
        a.send(0)
    for pr in procs:
        pr.join(timeout=5)
    value = per * cores * inner * args.steps / wall
    sample = ("%d reference RevoltFinal objects (%s) x %d env-steps per bench step, %d bench steps, %d persistent processes; "
              "simulator = the float64 stand-in twin" % (per * cores, ref_loader.source(), inner, args.steps, cores))
    port_val, _, port_sample = cpu_env_steps_per_s(1 << 16, 8)
    emit({
        "impl": "reference", "metric": "env_steps_per_sec", "value": value, "unit": "env-steps/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * wall / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(args, world),
        "cpu_baseline": {"value": value, "unit": "env-steps/s", "cores": cores, "kind": "reference", "sample": sample,
                         "port": {"value": port_val, "unit": "env-steps/s", "kind": "port", "sample": port_sample}},
        "e2e": {"value": value, "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    })


def workload_config(args, world):
    return {"workload": "BASELINE configs[2]: RevoltFinal(extended_state, cont_ang) env step, 3-DOF stand-in hull "
                        "x20 sub-steps, obs/reward/termination, auto-reset, random actions",
            "envs_per_gpu": args.envs_per_gpu, "global_envs": args.envs_per_gpu * world, "max_ep_len": 400,
            "n_substeps": 20, "parallelism": "env-sharded x%d, no collective" % world,
            "l2_policy": "inputs larger than L2 (per step: 1.0 GB state + 0.45 GB of fresh actions, a new window of a 2-buffer pool every step)"}


# ---- GPU side ----------------------------------------------------------------------------------------------------
def dump_outputs(path, obs, rew, done):
    """obs [9, n], reward [n] and the done flag byte [n] of one env step, on a fixed seeded sample of DUMP_ENVS
    environments (all of them when n is smaller), as float32; env_index.npy holds the sampled indices (float64)."""
    import numpy as np
    import torch
    n = rew.shape[0]
    idx = np.sort(np.random.default_rng(0).choice(n, min(n, DUMP_ENVS), replace=False))
    sel = torch.as_tensor(idx, device=obs.device)
    os.makedirs(path, exist_ok=True)
    for name, a in (("obs", obs[:, sel]), ("reward", rew[sel]), ("done", done[sel])):
        np.save(os.path.join(path, name + ".npy"), a.cpu().numpy().astype(np.float32))
    np.save(os.path.join(path, "env_index.npy"), idx.astype(np.float64))


def bind_to_gpu_cpus(index):
    """Multi-rank runs: pin this process to the CPUs NVML reports as local to its GPU, BEFORE the pinned host buffers of the
    end-to-end leg are allocated (first touch puts them on that NUMA node).  The launcher does not bind ranks, and eight
    ranks streaming 1.16 GB per step each through remote memory share the inter-socket link."""
    if os.environ.get("ML4CA_NO_BIND"):
        return "not bound (ML4CA_NO_BIND)"
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        words = (os.cpu_count() + 63) // 64
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, words)
        cpus = {64 * w + b for w, m in enumerate(mask) for b in range(64) if (m >> b) & 1}
        cpus &= set(os.sched_getaffinity(0))
        if cpus:
            os.sched_setaffinity(0, cpus)
            return "bound to %d CPUs local to GPU %d" % (len(cpus), index)
        return "not bound (empty NVML affinity)"
    except Exception as e:  # noqa: BLE001
        return "not bound (%r)" % (e,)


def run_b200(args, rank, local_rank, world):
    import torch
    import torch.distributed as dist
    from ml4ca_b200 import _lib
    from ml4ca_b200.env import RevoltFinal, StandInHull
    import ml4ca_b200 as M

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; this framework has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    numa_note = bind_to_gpu_cpus(local_rank) if world > 1 else "not bound (single rank)"
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    n = args.envs_per_gpu
    peak_gbs, peak_src = load_peaks()
    env = RevoltFinal(StandInHull(), extended_state=True, cont_ang=True, num_envs=n, device=dev, seed=2,
                      auto_reset=True, env_id_offset=rank * n)
    env.reset(fraction=0.8)
    gen = torch.Generator(device=dev)
    gen.manual_seed(2 + rank)
    room = ACTION_SHIFT * ((max(args.steps, 16) + 200 + args.warmup) // ACTION_POOL + 2)
    flat = [torch.rand(7 * n + room, device=dev, generator=gen) * 2 - 1 for _ in range(ACTION_POOL)]

    def actions(i):
        """Fresh a ~ U(-1,1)^7 for every (env, step): window i of the flat pools (no generation kernel in the timed loop)."""
        off = ACTION_SHIFT * ((i // ACTION_POOL) % (room // ACTION_SHIFT))
        return flat[i % ACTION_POOL][off:off + 7 * n].view(7, n)
    out = (torch.empty(9, n, device=dev), torch.empty(n, device=dev), torch.empty(n, dtype=torch.uint8, device=dev))

    sampler = ClockSampler(local_rank)
    sampler.start()

    # ---- device-resident timing ------------------------------------------------------------------------------
    for i in range(args.warmup):
        env.step_into(actions(i), *out)
    barrier()
    launches0 = _lib.launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sampler.mark("start")
    ev0.record()
    for i in range(args.steps):
        env.step_into(actions(args.warmup + i), *out)
    ev1.record()
    torch.cuda.synchronize()
    sampler.mark("end")
    ms = ev0.elapsed_time(ev1)
    launches = _lib.launch_count() - launches0
    if args.dump_outputs and rank == 0:        # before the sustained leg below overwrites `out`
        dump_outputs(args.dump_outputs, *out)
    barrier()
    ms_all = max_over_ranks(ms)
    ms_per_step = ms_all / args.steps
    value = n * world * args.steps / (ms_all * 1e-3)
    kernel_ms = ms / args.steps
    achieved = ENV_STEP_BYTES * n / (kernel_ms * 1e-3) / 1e9

    # ---- sustained leg: 200 back-to-back launches (the driver's 20-step run ends before the clock and the restart rate settle)
    sustained_ms = None
    if not args.skip_extra:
        sus = 200
        ev0.record()
        for i in range(sus):
            env.step_into(actions(args.warmup + args.steps + i), *out)
        ev1.record()
        torch.cuda.synchronize()
        sustained_ms = max_over_ranks(ev0.elapsed_time(ev1)) / sus

    # ---- end to end through the public API with host buffers ----------------------------------------------------
    e2e_steps = max(3, min(args.steps, 10))
    h_act = [(torch.rand(7, n) * 2 - 1).pin_memory() for _ in range(2)]
    h_obs = torch.empty(9, n).pin_memory()
    h_rew = torch.empty(n).pin_memory()
    h_done = torch.empty(n, dtype=torch.uint8).pin_memory()

    def e2e_step(i):
        # public API with host buffers: RevoltFinal.step_host -> ml4ca_env_step_host (chunked copy/compute pipeline)
        env.step_host(h_act[i % 2], h_obs, h_rew, h_done)

    for i in range(2):
        e2e_step(i)
    barrier()
    ev0.record()                      # step_host makes the caller's stream wait for the last result bytes, so events on
    for i in range(e2e_steps):        # this stream bracket copies in, kernels and copies out
        e2e_step(i)
    ev1.record()
    torch.cuda.synchronize()
    e2e_s = max_over_ranks(ev0.elapsed_time(ev1) * 1e-3)
    e2e_value = n * world * e2e_steps / e2e_s
    h2d = 7 * n * 4
    d2h = (9 * 4 + 4 + 1) * n
    # plain-copy ceiling of this box at this rank count: the same bytes per step, both directions at once, no kernel,
    # no chunking (one cudaMemcpyAsync per buffer on two streams).  e2e / ceiling says whether the pipeline or the box limits.
    d_act, d_out = torch.empty(7, n, device=dev), torch.empty(d2h, dtype=torch.uint8, device=dev)
    h_out = torch.empty(d2h, dtype=torch.uint8).pin_memory()
    s_in, s_out = torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev)

    def copy_step(i):
        with torch.cuda.stream(s_in):
            d_act.copy_(h_act[i % 2], non_blocking=True)
        with torch.cuda.stream(s_out):
            h_out.copy_(d_out, non_blocking=True)

    copy_step(0)
    barrier()
    c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    c0.record()
    s_in.wait_event(c0), s_out.wait_event(c0)
    for i in range(e2e_steps):
        copy_step(i)
    e_in, e_out = torch.cuda.Event(), torch.cuda.Event()
    e_in.record(s_in), e_out.record(s_out)
    torch.cuda.current_stream().wait_event(e_in), torch.cuda.current_stream().wait_event(e_out)
    c1.record()
    torch.cuda.synchronize()
    ceil_s = max_over_ranks(c0.elapsed_time(c1) * 1e-3)
    copy_ceiling = n * world * e2e_steps / ceil_s
    del d_act, d_out, h_out

    # ---- secondary kernels (rank-local, reported under "extra") -------------------------------------------------
    extra = {}
    try:
        m = 1 << 20
        eta = (torch.rand(3, m, device=dev, generator=gen) * 2 - 1) * torch.tensor([[8.0], [8.0], [0.785]], device=dev)
        nu = (torch.rand(3, m, device=dev, generator=gen) * 2 - 1) * torch.tensor([[1.4], [0.3], [0.52]], device=dev)
        ref = torch.zeros(3, m, device=dev)
        integ = torch.zeros(3, m, device=dev)
        for _ in range(3):
            M.pinv_pid(eta, nu, ref, integ)
        torch.cuda.synchronize()
        reps = 50
        ev0.record()
        for _ in range(reps):
            M.pinv_pid(eta, nu, ref, integ)
        ev1.record()
        torch.cuda.synchronize()
        t = ev0.elapsed_time(ev1) / reps * 1e-3
        extra["pinv_pid"] = {"workload": "BASELINE configs[1]: pseudoinverse + PID, 1 Mi setpoints (fits L2: "
                                         "an L2-resident figure, not an HBM one)",
                             "value": m / t, "unit": "allocations/s", "us_per_launch": t * 1e6,
                             "achieved_GBs": PINV_PID_BYTES * m / t / 1e9}
        m16 = 1 << 24                       # HBM-sized batch: 1.3 GB of rows per launch
        eta16 = (torch.rand(3, m16, device=dev, generator=gen) * 2 - 1) * torch.tensor([[8.0], [8.0], [0.785]], device=dev)
        nu16 = (torch.rand(3, m16, device=dev, generator=gen) * 2 - 1) * torch.tensor([[1.4], [0.3], [0.52]], device=dev)
        ref16, integ16 = torch.zeros(3, m16, device=dev), torch.zeros(3, m16, device=dev)
        for _ in range(3):
            M.pinv_pid(eta16, nu16, ref16, integ16)
        torch.cuda.synchronize()
        ev0.record()
        for _ in range(20):
            M.pinv_pid(eta16, nu16, ref16, integ16)
        ev1.record()
        torch.cuda.synchronize()
        t16 = ev0.elapsed_time(ev1) / 20 * 1e-3
        extra["pinv_pid_16Mi"] = {"workload": "pseudoinverse + PID, 16 Mi setpoints (1.3 GB of rows: an HBM figure)",
                                  "value": m16 / t16, "unit": "allocations/s", "ms_per_launch": t16 * 1e3,
                                  "achieved_GBs": PINV_PID_BYTES * m16 / t16 / 1e9,
                                  "hbm_frac": PINV_PID_BYTES * m16 / t16 / 1e9 / peak_gbs}
        del eta16, nu16, ref16, integ16
    except Exception as e:  # noqa: BLE001
        extra["pinv_pid"] = {"error": repr(e)}

    def timed(fn, reps, warm=2):
        for _ in range(warm):
            fn()
        torch.cuda.synchronize()
        ev0.record()
        for _ in range(reps):
            fn()
        ev1.record()
        torch.cuda.synchronize()
        return ev0.elapsed_time(ev1) / reps * 1e-3

    if not args.skip_extra:
        # K1: QP thrust allocation (BASELINE configs[0] batch law, SURVEY 8d config 1), 1 Mi demands
        try:
            import numpy as np
            from ml4ca_b200 import synth
            m = 1 << 20
            tau_np, prev_np = synth.qp_batch(4096, seed=0)
            reps_t = m // 4096
            tau_t = torch.as_tensor(np.tile(tau_np, reps_t), dtype=torch.float32, device=dev).contiguous()
            qp = M.QPTA(num_envs=m, device=dev)
            qp.previous_thruster_state = np.tile(prev_np, reps_t)
            barrier()
            t = max_over_ranks(timed(lambda: qp.solve_QP(tau_t), 5))
            extra["qp_allocate"] = {"workload": "BASELINE configs[0] demand law tiled to 1 Mi allocations per GPU (QPTA.solve_QP), "
                                                "SLSQP path in float64, aggregate over all ranks",
                                    "value": m * world / t, "unit": "allocations/s", "ms_per_launch": t * 1e3, "dtype": "f64",
                                    "achieved_GBs": QP_BYTES * m / t / 1e9, "hbm_frac": QP_BYTES * m / t / 1e9 / peak_gbs,
                                    "bound": "issue (FP64 pipe + divergence inside the active-set loops)"}
            del qp, tau_t
        except Exception as e:  # noqa: BLE001
            extra["qp_allocate"] = {"error": repr(e)}
        # K4: actor/critic 64x64 forward (configs[3]) stand-alone, and the rollout step built on it (policy kernel + env kernel)
        try:
            m = 1 << 23
            ac = M.ActorCritic(9, 7, (64, 64), "leaky_relu", device=dev, seed=3)
            obs_t = torch.rand(9, m, device=dev, generator=gen) * 2 - 1
            outp = (torch.empty(7, m, device=dev), torch.empty(m, device=dev), torch.empty(m, device=dev))
            t = timed(lambda: ac.step(obs_t, out=outp), 10)
            flop = 19712.0
            extra["policy_forward"] = {"workload": "BASELINE configs[3] network: 9-64-64-7 + 9-64-64-1 leaky-ReLU actor/critic, "
                                                   "8 Mi observations, tcgen05 fp16 operands / fp32 TMEM accumulators",
                                       "value": m / t, "unit": "observations/s", "ms_per_launch": t * 1e3,
                                       "achieved_GBs": POLICY_BYTES * m / t / 1e9, "achieved_TFLOPs": flop * m / t / 1e12,
                                       "roofline": {"bound": "tensor", "achieved": flop * m / t / 1e12, "peak": load_tensor_peak()[0],
                                                    "unit": "TFLOP/s", "frac": flop * m / t / 1e12 / load_tensor_peak()[0],
                                                    "peak_source": load_tensor_peak()[1],
                                                    "note": "algorithmic flop (19 712 per observation); tensor pipe 64 % active under ncu "
                                                            "(profiles/policy_qp_r1.md): the MMAs are operand-read bound"}}
            env2 = RevoltFinal(StandInHull(), extended_state=True, cont_ang=True, num_envs=m, device=dev, seed=4,
                               auto_reset=True, env_id_offset=rank * m)
            env2.reset(fraction=0.8)
            buf = M.TrajectoryBuffer(9, 7, 32, m, device=dev)     # 32 steps per call: the per-window bootstrap forward (ppo.py:311) is 1 / 32 of a policy pass
            state = {"t": 0}

            def roll():
                M.rollout(env2, ac, buf, seed=3, start_step=state["t"])
                state["t"] += buf.max_size
            t = timed(roll, 3, warm=1) / buf.max_size
            extra["rollout_two_kernel"] = {
                "workload": "configs[3]: policy forward + env step + trajectory record, 8 Mi envs/GPU, training mode "
                            "(one policy kernel + one env kernel per step; fused arrangements measured slower: profiles/rollout_r2.md)",
                "value": m / t, "unit": "env-steps/s", "ms_per_step": t * 1e3,
                "achieved_GBs": ROLLOUT_TRAIN_BYTES * m / t / 1e9}
            # K5: GAE-lambda over the [T, n] buffer
            Tg = 64
            mg = 1 << 21
            gbuf = M.TrajectoryBuffer(1, 1, Tg, mg, gamma=0.99, lam=0.97, device=dev)
            gbuf.rew_buf.normal_(generator=gen); gbuf.val_buf.normal_(generator=gen)
            t = timed(lambda: gbuf.finish_path(), 5)
            extra["gae"] = {"workload": "TrajectoryBuffer.finish_path, T=64 x 2 Mi envs", "value": Tg * mg / t,
                            "unit": "steps/s", "ms_per_launch": t * 1e3, "achieved_GBs": GAE_BYTES * Tg * mg / t / 1e9,
                            "hbm_frac": GAE_BYTES * Tg * mg / t / 1e9 / peak_gbs}
            del env2, buf, gbuf, ac
        except Exception as e:  # noqa: BLE001
            extra["policy_rollout"] = {"error": repr(e)}

    if not args.skip_extra:
        # config 5: full PPO training (rollout, GAE, update with the gradient all-reduce over all ranks)
        try:
            ne, Tp = 1 << 14, 400
            env3 = RevoltFinal(StandInHull(), extended_state=True, cont_ang=True, num_envs=ne, device=dev, seed=5,
                               auto_reset=True, env_id_offset=rank * ne)
            ac3 = M.ActorCritic(9, 7, (64, 64), "leaky_relu", device=dev, seed=5)
            # one run of 5 epochs: the first two warm up (parameter sync, eager rollout, graph capture), the median of the last three is reported
            marks = []

            def mark(info):
                torch.cuda.synchronize()
                marks.append(time.perf_counter())
            _, hist = M.ppo(env3, ac3, steps_per_epoch=Tp, epochs=5, seed=5, graph=True, logger=mark)
            dt = max_over_ranks(sorted(b - a for a, b in zip(marks[1:-1], marks[2:]))[1])     # median of the last three epochs
            hist = hist[2:]
            passes = sum(h["StopIter"] + 1 + 80 + 2 for h in hist) / float(len(hist))
            extra["ppo_train"] = {"workload": "BASELINE configs[4]: PPO epoch = 400-step rollout of 16 Ki envs/GPU + GAE + update "
                                              "(config.json hyper-parameters: <= 80 pi + 80 v full-batch Adam iterations, target_kl 0.01), "
                                              "NCCL all-reduce of the flat gradient per iteration; rollout replayed from a CUDA graph",
                                  "value": ne * world * Tp / dt, "unit": "env-steps/s incl. update", "s_per_epoch": dt,
                                  "gradient_passes_per_epoch": passes,
                                  "sample_passes_per_s": passes * ne * world * Tp / dt, "last_epoch": {k: hist[-1][k] for k in ("StopIter", "KL", "LossV", "AverageStepReward")}}
            del env3, ac3
        except Exception as e:  # noqa: BLE001
            extra["ppo_train"] = {"error": repr(e)}
        # the same training loop with the reference's OWN default network (train.py:30-32: 80 x 80 x 80, every shipped checkpoint but
        # one): tcgen05 forward and tcgen05 gradient kernel (csrc/ppo_update_tc.cu templated on width and depth), same batch as above
        try:
            ne, Tp = 1 << 14, 400
            env4 = RevoltFinal(StandInHull(), extended_state=True, cont_ang=True, num_envs=ne, device=dev, seed=6,
                               auto_reset=True, env_id_offset=rank * ne)
            ac4 = M.ActorCritic(9, 7, (80, 80, 80), "leaky_relu", device=dev, seed=6)
            marks = []

            def mark4(info):
                torch.cuda.synchronize()
                marks.append(time.perf_counter())
            _, hist = M.ppo(env4, ac4, steps_per_epoch=Tp, epochs=4, seed=6, graph=True, logger=mark4)
            dt = max_over_ranks(sorted(b - a for a, b in zip(marks[1:-1], marks[2:]))[0])
            hist = hist[2:]
            passes = sum(h["StopIter"] + 1 + 80 + 2 for h in hist) / float(len(hist))
            extra["ppo_train_80x3"] = {"workload": "PPO epoch with the reference's default 80 x 80 x 80 network, 16 Ki envs/GPU x 400 steps "
                                                   "(tcgen05 forward and gradient kernels, one tile group per CTA at this width)",
                                       "value": ne * world * Tp / dt, "unit": "env-steps/s incl. update", "s_per_epoch": dt,
                                       "gradient_passes_per_epoch": passes, "sample_passes_per_s": passes * ne * world * Tp / dt}
            del env4, ac4
        except Exception as e:  # noqa: BLE001
            extra["ppo_train_80x3"] = {"error": repr(e)}
        # the same epoch with the TRPO update (train.py --algo trpo): CG on the Fisher-vector product + line search + 80 v steps;
        # once with every policy pass on the fp32 kernel (parity mode, default) and once with the CG passes on tcgen05
        for leg, kern in (("trpo_train", "fp32"), ("trpo_train_tc", "tensor_core")):
            try:
                ne, Tp = 1 << 14, 400
                env4 = RevoltFinal(StandInHull(), extended_state=True, cont_ang=True, num_envs=ne, device=dev, seed=7,
                                   auto_reset=True, env_id_offset=rank * ne)
                ac4 = M.ActorCritic(9, 7, (64, 64), "leaky_relu", device=dev, seed=7)
                marks = []

                def mark4(info):
                    torch.cuda.synchronize()
                    marks.append(time.perf_counter())
                _, hist = M.trpo(env4, ac4, steps_per_epoch=Tp, epochs=5, seed=7, graph=True, logger=mark4, kernel=kern)
                dt = max_over_ranks(sorted(b - a for a, b in zip(marks[1:-1], marks[2:]))[1])
                extra[leg] = {"workload": "TRPO epoch = 400-step rollout of 16 Ki envs/GPU + GAE + update (trpo.py defaults: "
                                          "10 CG iterations on the damped Fisher-vector product, <= 10 backtracking steps, "
                                          "80 v iterations), all-reduce of every flat gradient; KL-gradient passes of the CG solve on the "
                                          + ("fp32 CUDA-core kernel" if kern == "fp32" else "tcgen05 kernel"),
                              "value": ne * world * Tp / dt, "unit": "env-steps/s incl. update", "s_per_epoch": dt,
                              "last_epoch": {k: hist[-1][k] for k in ("KL", "BacktrackIters", "DeltaLossPi", "LossV")}}
                del env4, ac4
            except Exception as e:  # noqa: BLE001
                extra[leg] = {"error": repr(e)}

    sampler.stop_flag.set()
    sampler.join(timeout=1.0)
    clocks = sampler.summary()

    if rank == 0:
        cpu_kind, cpu_port = "port", None
        if args.skip_cpu:
            cpu_val, cpu_cores, cpu_sample = None, 0, "skipped (--skip-cpu)"
        else:
            cpu_val, cpu_cores, cpu_sample = cpu_env_steps_per_s(1 << 16, 8)
            if reference_code_available():          # the reference's own code is on the box: it is the baseline, the port is a note
                cpu_port = {"value": cpu_val, "unit": "env-steps/s", "cores": cpu_cores, "kind": "port", "sample": cpu_sample}
                cpu_val, cpu_cores, cpu_sample = refcode_env_steps_per_s(8, 100)
                cpu_kind = "reference"
            try:
                if "qp_allocate" in extra and "error" not in extra["qp_allocate"]:
                    extra["qp_allocate"]["cpu_baseline"] = cpu_qp_allocations_per_s(512)
                one = cpu_env_steps_per_s(1 << 13, 8, cores=1)
                extra["cpu_env_single_core"] = {"value": one[0], "unit": "env-steps/s", "cores": 1, "sample": one[2]}
            except Exception as e:  # noqa: BLE001
                extra["cpu_baselines_error"] = repr(e)
        # compact per-kernel figures inside the object the driver keeps (BASELINE's metric names env-steps/s AND QP allocations/s)
        kernels = {}

        def pick(name, keys):
            e = extra.get(name)
            if isinstance(e, dict) and "error" not in e:
                kernels[name] = {k: e[k] for k in keys if k in e}
        pick("qp_allocate", ("value", "unit", "ms_per_launch", "dtype", "hbm_frac", "bound"))
        if "qp_allocate" in kernels and isinstance(extra["qp_allocate"].get("cpu_baseline"), dict):
            cb = extra["qp_allocate"]["cpu_baseline"]
            kernels["qp_allocate"]["cpu_baseline"] = {k: cb[k] for k in ("value", "unit", "cores", "kind")}
        pick("pinv_pid", ("value", "unit", "us_per_launch"))
        pick("pinv_pid_16Mi", ("value", "unit", "ms_per_launch", "hbm_frac"))
        pick("policy_forward", ("value", "unit", "ms_per_launch", "achieved_TFLOPs"))
        for k in ("rollout_two_kernel",):
            pick(k, ("value", "unit", "ms_per_step", "achieved_GBs"))
            if k in kernels:
                kernels[k]["hbm_frac"] = kernels[k]["achieved_GBs"] / peak_gbs
        pick("gae", ("value", "unit", "ms_per_launch", "hbm_frac"))
        for k in ("ppo_train", "ppo_train_80x3", "trpo_train", "trpo_train_tc"):
            pick(k, ("value", "unit", "s_per_epoch", "sample_passes_per_s"))
        line = {
            "metric": "env_steps_per_sec", "value": value, "unit": "env-steps/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(args, world),
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak_gbs, "unit": "GB/s",
                         "frac": achieved / peak_gbs, "traffic": ENV_STEP_TRAFFIC, "peak_source": peak_src,
                         "traffic_source": "dram__bytes_read.sum + dram__bytes_write.sum, ncu --set full, profiles/env_step_r1.md",
                         "kernel": "env_step_kernel<FINAL,cont,ext,2 envs/thread>", "bytes_per_env_step": ENV_STEP_BYTES,
                         "kernel_ms": kernel_ms,
                         "sustained_ms": sustained_ms,
                         "sustained_frac": (ENV_STEP_BYTES * n / (sustained_ms * 1e-3) / 1e9 / peak_gbs) if sustained_ms else None,
                         "sustained_note": "200 further back-to-back launches (stationary clock and restart rate)",
                         "kernels": kernels},
            "cpu_baseline": dict({"value": cpu_val, "unit": "env-steps/s", "cores": cpu_cores, "kind": cpu_kind,
                                  "sample": cpu_sample}, **({"port": cpu_port} if cpu_port else {})),
            "e2e": {"value": e2e_value, "unit": "env-steps/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "steps": e2e_steps, "copy_ceiling": copy_ceiling, "frac_of_copy_ceiling": e2e_value / copy_ceiling,
                    "copy_ceiling_note": "same bytes per step, pinned host <-> device both ways at once, no kernel, measured at this rank count in this run",
                    "note": "RevoltFinal.step_host: pinned host actions in, obs+reward+done out, every step, chunked H2D|kernel|D2H pipeline",
                    "cpu_binding": numa_note},
            "gpu_launches": int(launches), "clocks": clocks, "extra": extra,
        }
        emit(line)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--envs-per-gpu", type=int, default=1 << 24)
    ap.add_argument("--skip-cpu", action="store_true", help="omit the CPU baseline leg (used for ncu captures)")
    ap.add_argument("--skip-extra", action="store_true", help="omit the secondary-kernel figures under 'extra'")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the outputs of the last timed step (obs, reward, done of a fixed env sample) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the b200 path")
    args.warmup = max(args.warmup, 3)
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    run_b200(args, rank, local_rank, world)


if __name__ == "__main__":
    main()
