"""First-order wave-frequency motion (ml4ca_env_set_waves): throughput of the WAVE step kernels and the controller
comparison in waves.  Writes profiles/waves_r3.md-style tables to stdout and the raw numbers as JSON (--out).

  (a) throughput: 16 Mi RevoltFinal envs (continuous angles, extended state), 200 steps per timed window, CUDA events; the
      default kernel, WAVE, WAVE + DIST with a Gauss-Markov bias (sigma_bias > 0) and DIST alone, timed alternately.
      Bytes per env-step: 177 (default) / 229 (WAVE) / 261 (WAVE + DIST) / 209 (DIST), over 6456.5 GB/s.
  (b) --bench-parent DIR: bench.py --gpus 1 --steps 200 of this tree and of the built tree DIR, alternately (3 runs each).
  (c) closed loop: the shipped 80^3 policy, the same with the deployment node's body-frame integrator, PID + QP and
      PID + pseudoinverse, from the 6 fixed test poses, sigma_pos in {0, 0.05, 0.1, 0.2} m in surge and sway,
      sigma_yaw = sigma_pos * 20 deg/m, w0 ~ U(1, 2) rad/s, lambda = 0.1, 400 steps, 8 seeds of the wave draws.
      The controllers see the measured pose; IAE scores the LF pose.
  (d) --train: PPO at the reference configuration (80^3, 4 envs x 400 steps, 800 epochs) in waves with sigma_pos = 0.1 m,
      then evaluated as in (c).
"""
import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

import ml4ca_b200 as M
from ml4ca_b200 import evaluate

HBM_GBS = 6456.5
SIGMAS = (0.0, 0.05, 0.1, 0.2)
SEEDS = 8


def sea(sigma_pos):
    return dict(sigma=(sigma_pos, sigma_pos, np.deg2rad(20.0 * sigma_pos)), peak_frequency=(1.0, 2.0), damping=0.1)


def gpu_line():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                              text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:      # the line is informative only
        return "unknown (%s)" % e


def throughput(dev, n, steps, reps):
    dist = dict(current_speed=(0.0, 0.2), current_direction=(0.0, 2 * np.pi), bias_std=(10.0, 10.0, 5.0), bias_time_s=30.0)
    variants = [("default", None, None, 177), ("WAVE", sea(0.1), None, 229), ("WAVE+DIST", sea(0.1), dist, 261),
                ("DIST", None, dist, 209)]
    g = torch.Generator(device=dev)
    g.manual_seed(0)
    act = torch.rand(7, n, device=dev, generator=g) * 2 - 1
    envs = []
    for name, waves, dist_kw, nbytes in variants:
        env = M.RevoltFinal(M.StandInHull(), extended_state=True, cont_ang=True, num_envs=n, device=dev, seed=1, auto_reset=True)
        if dist_kw is not None:
            env.set_disturbance(**dist_kw)
        if waves is not None:
            env.set_waves(**waves)
        env.reset()
        out = (torch.empty(9, n, device=dev), torch.empty(n, device=dev), torch.empty(n, dtype=torch.uint8, device=dev))
        for _ in range(20):                                              # warm-up
            env.step_into(act, *out)
        envs.append((name, env, out, nbytes))
    times = {name: [] for name, _, _, _ in envs}
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(reps):
        for name, env, out, _ in envs:
            torch.cuda.synchronize()
            e0.record()
            for _ in range(steps):
                env.step_into(act, *out)
            e1.record()
            e1.synchronize()
            times[name].append(e0.elapsed_time(e1) / steps)
    rows = []
    for name, _, _, nbytes in envs:
        ms = float(np.median(times[name]))
        rate = n / (ms * 1e-3)
        rows.append(dict(variant=name, ms_per_step=ms, spread_ms=[float(min(times[name])), float(max(times[name]))],
                         g_env_steps_per_s=rate / 1e9, bytes_per_env_step=nbytes,
                         hbm_fraction=rate * nbytes / (HBM_GBS * 1e9)))
    return rows


def bench_ab(parent, steps, runs):
    """bench.py --gpus 1 --steps <steps> of this tree and of ``parent``, alternately; the JSON headline of each run."""
    here = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = {"this": [], "parent": []}
    for _ in range(runs):
        for key, root in (("this", here), ("parent", parent)):
            p = subprocess.run([sys.executable, "bench.py", "--gpus", "1", "--steps", str(steps), "--warmup", "20"], cwd=root,
                               capture_output=True, text=True, timeout=1800)
            line = [l for l in p.stdout.splitlines() if l.startswith("{")]
            out[key].append(json.loads(line[-1]) if line else {"error": p.stderr[-2000:]})
    return out


def closed_loop(dev, controllers, steps):
    rows = []
    n = 6 * SEEDS
    calm = {}
    for sp in SIGMAS:
        for name, run in controllers:
            env = M.RevoltFinal(M.StandInHull(), testing=True, extended_state=True, cont_ang=True, num_envs=n, device=dev,
                                max_ep_len=2 * steps, seed=11)
            if sp > 0:
                env.set_waves(**sea(sp))
            rec = run(env)
            eta = rec["eta"].cpu().numpy()
            m = rec["metrics"].cpu().numpy()
            tail = eta[-100:]
            pos, yaw = np.hypot(tail[:, 0], tail[:, 1]).mean(axis=0), np.rad2deg(np.abs(tail[:, 2])).mean(axis=0)
            W = float(m[1].mean())
            if sp == 0:
                calm[name] = W
            rows.append(dict(sigma_pos=sp, controller=name, IAE=float(m[0].mean()), W=W, IADC=float(m[2].mean()),
                             W_increase=W / calm[name] - 1.0, pos_err_m=float(pos.mean()), yaw_err_deg=float(yaw.mean())))
            print("  %.2f m  %-14s IAE %8.2f  W* %8.1f (%+6.1f %%)  IADC %8.3f  |pos| %.3f m  |yaw| %.2f deg" % (
                sp, name, rows[-1]["IAE"], W, 100 * rows[-1]["W_increase"], rows[-1]["IADC"], rows[-1]["pos_err_m"],
                rows[-1]["yaw_err_deg"]), flush=True)
    return rows


def controllers_for(ac, steps):
    return [("RL", lambda env: evaluate.run_RL_policy(env, ac, max_ep_len=steps)),
            ("RL+integrator", lambda env: evaluate.run_RL_policy(env, ac, max_ep_len=steps, integrator=True)),
            ("QP", lambda env: evaluate.run_allocator(env, "qp", max_ep_len=steps)),
            ("pinv", lambda env: evaluate.run_allocator(env, "pinv", max_ep_len=steps))]


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--n", type=int, default=1 << 24)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--eval-steps", type=int, default=400)
    ap.add_argument("--skip-throughput", action="store_true")
    ap.add_argument("--skip-closed-loop", action="store_true")
    ap.add_argument("--bench-parent", default=None, help="(b): a built tree of the parent commit to run bench.py against")
    ap.add_argument("--bench-runs", type=int, default=3)
    ap.add_argument("--train", action="store_true", help="(d): PPO 80^3, 4 x 400, 800 epochs in waves, sigma_pos = 0.1 m")
    ap.add_argument("--epochs", type=int, default=800)
    ap.add_argument("--out", default=None, help="JSON file for the raw numbers")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("wave_eval.py needs a CUDA device")
    dev = torch.device("cuda", 0)
    res = {"gpu": gpu_line()}
    print("GPU, power limit:", res["gpu"], flush=True)
    if not args.skip_throughput:
        res["throughput"] = throughput(dev, args.n, args.steps, args.reps)
        print("(a) %d envs, %d steps per window, median of %d alternating windows" % (args.n, args.steps, args.reps))
        print("| variant | ms / step | G env-steps/s | B / env-step | of 6456.5 GB/s |\n|---|---|---|---|---|")
        for r in res["throughput"]:
            print("| %s | %.4f (%.4f-%.4f) | %.2f | %d | %.1f %% |" % (r["variant"], r["ms_per_step"], r["spread_ms"][0],
                                                                    r["spread_ms"][1], r["g_env_steps_per_s"],
                                                                    r["bytes_per_env_step"], 100 * r["hbm_fraction"]))
    if args.bench_parent:
        res["bench"] = bench_ab(args.bench_parent, args.steps, args.bench_runs)
        print("(b) bench.py --gpus 1 --steps %d, alternating this tree and the parent" % args.steps)
        for key in ("this", "parent"):
            print("  %-6s %s" % (key, json.dumps(res["bench"][key])), flush=True)
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    if not args.skip_closed_loop:
        params = np.load(os.path.join(root, "tests", "golden", "policy_final_80x3.npz"))["params"]
        ac = M.ActorCritic(9, 7, (80, 80, 80), "leaky_relu", params=params, device=dev)
        print("(c) shipped 80^3 policy, RL + integrator, QP, pinv; 6 poses x %d wave seeds, %d steps" % (SEEDS, args.eval_steps),
              flush=True)
        t0 = time.perf_counter()
        res["closed_loop"] = closed_loop(dev, controllers_for(ac, args.eval_steps), args.eval_steps)
        print("  (%.0f s)" % (time.perf_counter() - t0))
    if args.train:
        env = M.RevoltFinal(M.StandInHull(), extended_state=True, cont_ang=True, num_envs=4, device=dev, seed=0, auto_reset=True)
        env.set_waves(**sea(0.1))
        t0 = time.perf_counter()
        ac_t, hist = M.ppo(env, steps_per_epoch=400, epochs=args.epochs, seed=0, hidden_sizes=(80, 80, 80),
                           activation="leaky_relu", graph=True)
        torch.cuda.synchronize()
        secs = time.perf_counter() - t0
        last = hist[-20:]
        res["train"] = dict(seconds=secs, epochs=args.epochs,
                            last20_step_reward=float(np.mean([h["AverageStepReward"] for h in last])))
        print("(d) PPO 80^3, 4 x 400, %d epochs in waves (sigma_pos 0.1 m): %.1f s, mean step reward of the last 20 epochs %.3f"
              % (args.epochs, secs, res["train"]["last20_step_reward"]), flush=True)
        rl = [c for c in controllers_for(ac_t, args.eval_steps) if c[0].startswith("RL")]
        res["train"]["closed_loop"] = closed_loop(dev, rl, args.eval_steps)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()
