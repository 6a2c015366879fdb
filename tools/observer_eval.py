"""Passive nonlinear DP observer (ml4ca_observer_step): throughput of the observer kernel and the controller comparison in
waves with and without it.  Writes profiles/observer_r3.md-style tables to stdout and the raw numbers as JSON (--out).

  (a) throughput: 16 Mi envs, 200 back-to-back launches per timed window, CUDA events, 5 windows each: the observer step
      (hull 0, step_dt 0.2 s: 20 sub-steps) and the default env step (RevoltFinal, continuous angles, extended state) as the
      reference point, timed alternately.  Inputs and state are far larger than L2 (2.7 GB for the observer).
      Algorithmic bytes: 161 per observer step, 177 per env step, over 6456.5 GB/s.
  (b) closed loop: the sea states, seeds and controllers of tools/wave_eval.py (c) -- the shipped 80^3 policy, the same with
      the deployment node's integrator, PID + QP and PID + pseudoinverse, 6 fixed poses x 8 wave seeds, 400 steps -- each
      without an observer, with an observer at w_o = 1.5 rad/s fixed, and with w_o = the env's true w0.
  (c) bias estimation: waves (sigma_pos 0.1 m) plus the disturbance with current 0, bias sigma (10 N, 10 N, 5 Nm) and
      T_b = 30 s, PID + pseudoinverse on the observer (true w0): RMS of b^ - b over the last 200 of 400 steps.
  (d) --bench-parent DIR: bench.py --gpus 1 --steps 200 of this tree and of the built tree DIR, alternately.
"""
import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import numpy as np
import torch

import ml4ca_b200 as M
import wave_eval as WE
from ml4ca_b200 import evaluate

HBM_GBS = WE.HBM_GBS
OBS_BYTES, ENV_BYTES = 161, 177


def throughput(dev, n, steps, reps):
    g = torch.Generator(device=dev)
    g.manual_seed(0)
    act = torch.rand(7, n, device=dev, generator=g) * 2 - 1
    env = M.RevoltFinal(M.StandInHull(), extended_state=True, cont_ang=True, num_envs=n, device=dev, seed=1, auto_reset=True)
    env.reset()
    out = (torch.empty(9, n, device=dev), torch.empty(n, device=dev), torch.empty(n, dtype=torch.uint8, device=dev))
    obs = M.DPObserver(n, device=dev)
    y = torch.rand(3, n, device=dev, generator=g) * 2 - 1
    thrust = torch.rand(3, n, device=dev, generator=g) * 200 - 100
    angles = torch.rand(3, n, device=dev, generator=g) * 6 - 3
    obs.omega_o.uniform_(1.0, 2.0, generator=g)
    obs.reset(y)
    runs = [("observer_step_kernel", lambda: obs.step(y, thrust, angles), OBS_BYTES),
            ("env step (default kernel)", lambda: env.step_into(act, *out), ENV_BYTES)]
    for _, fn, _ in runs:
        for _ in range(20):                                              # warm-up
            fn()
    times = {name: [] for name, _, _ in runs}
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(reps):
        for name, fn, _ in runs:
            torch.cuda.synchronize()
            e0.record()
            for _ in range(steps):
                fn()
            e1.record()
            e1.synchronize()
            times[name].append(e0.elapsed_time(e1) / steps)
    assert torch.isfinite(obs.state).all()
    rows = []
    for name, _, nbytes in runs:
        ms = float(np.median(times[name]))
        rate = n / (ms * 1e-3)
        rows.append(dict(kernel=name, ms_per_step=ms, spread_ms=[float(min(times[name])), float(max(times[name]))],
                         g_steps_per_s=rate / 1e9, bytes_per_env_step=nbytes, hbm_fraction=rate * nbytes / (HBM_GBS * 1e9),
                         hbm_floor_ms=n * nbytes / (HBM_GBS * 1e9) * 1e3))
    return rows


def make_observer(mode, env):
    if mode == "none":
        return None
    ob = M.DPObserver.for_env(env)
    if mode == "true w0":                  # the run's own env reset draws w0: read it when the run resets the observer
        reset = ob.reset

        def reset_true(y, mask=None):
            ob.omega_o.copy_(env.get_state()["wave_omega"])
            reset(y, mask)
        ob.reset = reset_true
    return ob


def closed_loop(dev, ac, steps):
    runs = [("RL", lambda env, ob: evaluate.run_RL_policy(env, ac, max_ep_len=steps, observer=ob)),
            ("RL+integrator", lambda env, ob: evaluate.run_RL_policy(env, ac, max_ep_len=steps, integrator=True, observer=ob)),
            ("QP", lambda env, ob: evaluate.run_allocator(env, "qp", max_ep_len=steps, observer=ob)),
            ("pinv", lambda env, ob: evaluate.run_allocator(env, "pinv", max_ep_len=steps, observer=ob))]
    n = 6 * WE.SEEDS
    rows, calm = [], {}
    for sp in WE.SIGMAS:
        for name, run in runs:
            for mode in ("none", "w_o 1.5", "true w0"):
                if sp == 0 and mode == "true w0":
                    continue                                             # no waves, no true w0
                env = M.RevoltFinal(M.StandInHull(), testing=True, extended_state=True, cont_ang=True, num_envs=n,
                                    device=dev, max_ep_len=2 * steps, seed=11)
                if sp > 0:
                    env.set_waves(**WE.sea(sp))
                rec = run(env, make_observer(mode, env))
                eta = rec["eta"].cpu().numpy()
                m = rec["metrics"].cpu().numpy()
                tail = eta[-100:]
                pos, yaw = np.hypot(tail[:, 0], tail[:, 1]).mean(axis=0), np.rad2deg(np.abs(tail[:, 2])).mean(axis=0)
                W = float(m[1].mean())
                if sp == 0 and mode == "none":
                    calm[name] = W
                rows.append(dict(sigma_pos=sp, controller=name, observer=mode, IAE=float(m[0].mean()), W=W,
                                 IADC=float(m[2].mean()), W_over_calm=W / calm[name], pos_err_m=float(pos.mean()),
                                 yaw_err_deg=float(yaw.mean())))
                r = rows[-1]
                print("| %.2f | %s | %s | %.2f | %.1f | %.2f | %.3f | %.4f | %.3f |" % (
                    sp, name, mode, r["IAE"], W, r["W_over_calm"], r["IADC"], r["pos_err_m"], r["yaw_err_deg"]), flush=True)
    return rows


def bias_estimation(dev, steps):
    n = 6 * WE.SEEDS
    env = M.RevoltFinal(M.StandInHull(), testing=True, extended_state=True, cont_ang=True, num_envs=n, device=dev,
                        max_ep_len=2 * steps, seed=11)
    env.set_disturbance(current_speed=(0.0, 0.0), bias_std=(10.0, 10.0, 5.0), bias_time_s=30.0)
    env.set_waves(**WE.sea(0.1))
    ob = make_observer("true w0", env)
    trace = []
    step = ob.step

    def recording_step(y, thrust, angles, restart=None):
        out = step(y, thrust, angles, restart)
        trace.append((ob.bias_hat.clone(), env.get_state()["bias"]))
        return out
    ob.step = recording_step
    rec = evaluate.run_allocator(env, "pinv", max_ep_len=steps, observer=ob)
    est = torch.stack([t[0] for t in trace]).cpu().numpy()[-200:]
    true = torch.stack([t[1] for t in trace]).cpu().numpy()[-200:]
    rms = np.sqrt(((est - true) ** 2).mean(axis=(0, 2)))
    std = np.sqrt((true ** 2).mean(axis=(0, 2)))
    return dict(rms_error=rms.tolist(), rms_true=std.tolist(), IAE=float(rec["metrics"][0].mean()),
                W=float(rec["metrics"][1].mean()))


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--n", type=int, default=1 << 24)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--eval-steps", type=int, default=400)
    ap.add_argument("--skip-throughput", action="store_true")
    ap.add_argument("--skip-closed-loop", action="store_true")
    ap.add_argument("--bench-parent", default=None, help="(d): a built tree of the parent commit to run bench.py against")
    ap.add_argument("--bench-runs", type=int, default=3)
    ap.add_argument("--out", default=None, help="JSON file for the raw numbers")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("observer_eval.py needs a CUDA device")
    dev = torch.device("cuda", 0)
    res = {"gpu": WE.gpu_line()}
    print("GPU, power limit:", res["gpu"], flush=True)
    if not args.skip_throughput:
        res["throughput"] = throughput(dev, args.n, args.steps, args.reps)
        print("(a) %d envs, %d launches per window, median (range) of %d alternating windows" % (args.n, args.steps, args.reps))
        print("| kernel | ms / step | G steps/s | B / env-step | HBM floor ms | of 6456.5 GB/s |\n|---|---|---|---|---|---|")
        for r in res["throughput"]:
            print("| %s | %.4f (%.4f-%.4f) | %.2f | %d | %.3f | %.1f %% |" % (
                r["kernel"], r["ms_per_step"], r["spread_ms"][0], r["spread_ms"][1], r["g_steps_per_s"],
                r["bytes_per_env_step"], r["hbm_floor_ms"], 100 * r["hbm_fraction"]), flush=True)
    if not args.skip_closed_loop:
        params = np.load(os.path.join(ROOT, "tests", "golden", "policy_final_80x3.npz"))["params"]
        ac = M.ActorCritic(9, 7, (80, 80, 80), "leaky_relu", params=params, device=dev)
        print("(b) 6 poses x %d wave seeds, %d steps" % (WE.SEEDS, args.eval_steps), flush=True)
        print("| sigma_pos m | controller | observer | IAE | W* | W* / calm | IADC | LF pos err m | LF yaw err deg |\n"
              "|---|---|---|---|---|---|---|---|---|")
        t0 = time.perf_counter()
        res["closed_loop"] = closed_loop(dev, ac, args.eval_steps)
        print("  (%.0f s)" % (time.perf_counter() - t0))
        res["bias"] = bias_estimation(dev, args.eval_steps)
        print("(c) bias estimation, RMS of b^ - b over the last 200 steps (N, N, Nm): %s; RMS of b: %s" % (
            np.round(res["bias"]["rms_error"], 3).tolist(), np.round(res["bias"]["rms_true"], 3).tolist()), flush=True)
    if args.bench_parent:
        res["bench"] = WE.bench_ab(args.bench_parent, args.steps, args.bench_runs)
        print("(d) bench.py --gpus 1 --steps %d, alternating this tree and the parent" % args.steps)
        for key in ("this", "parent"):
            print("  %-6s %s" % (key, json.dumps(res["bench"][key])), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()
