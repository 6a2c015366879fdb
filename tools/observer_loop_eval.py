"""DP observer in the loop (ml4ca_env_set_observer, the OBSV step kernels): throughput, epoch times and the training
experiment of profiles/observer_loop_r3.md.  Prints the tables and writes the raw numbers as JSON (--out).

  (a) throughput at 16 Mi envs (RevoltFinal, extended state, continuous angles), 200 back-to-back steps per timed window,
      CUDA events, 5 alternating windows: the step, the step with the observer in the loop, and the step followed by
      ml4ca_observer_step plus the copy of the three nu^ rows into the observation (what a two-kernel rollout would
      launch), each with and without waves.  Bytes per env-step: 177 / 229 (waves), + 124 fused, + 161 + 24 two-kernel.
  (b) --bench-parent DIR: bench.py --gpus 1 --steps 200 of this tree and of the built tree DIR, alternately.
  (c) one graph-replayed PPO epoch (80^3, leaky-ReLU) with and without an attached observer, at 4 x 400 and 16 Ki x 400.
  (d) the hypothesis: PPO with the reference configuration (80^3, 4 envs x 400 steps, graph-replayed) in waves
      sigma = (0.1 m, 0.1 m, 2 deg), w0 ~ U(1, 2), lambda = 0.1, arm A on the measured observation, arm B with an observer
      attached (w_o = 1.5 rad/s); both evaluated through run_RL_policy with a separate observer (w_o = 1.5) on a plain env,
      6 fixed poses x 8 seeds, 400 steps, at sigma_pos 0, 0.05, 0.1, 0.2 m.
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
SEA = WE.sea(0.1)


def make_env(dev, n, waves, **kw):
    env = M.RevoltFinal(M.StandInHull(), extended_state=True, cont_ang=True, num_envs=n, device=dev, **kw)
    if waves:
        env.set_waves(**SEA)
    return env


def throughput(dev, n, steps, reps):
    g = torch.Generator(device=dev)
    g.manual_seed(0)
    act = torch.rand(7, n, device=dev, generator=g) * 2 - 1
    y = torch.rand(3, n, device=dev, generator=g) * 2 - 1              # the two-kernel sequence reads the measured pose,
    thrust = torch.rand(3, n, device=dev, generator=g) * 200 - 100      # thrust and azimuths from rows of their own
    angles = torch.rand(3, n, device=dev, generator=g) * 6 - 3
    runs = []
    for waves in (False, True):
        base = 229 if waves else 177
        tag = " + waves" if waves else ""
        for mode in ("step", "fused", "two-kernel"):
            env = make_env(dev, n, waves, seed=1, auto_reset=True)
            env.reset()
            out = (torch.empty(9, n, device=dev), torch.empty(n, device=dev), torch.empty(n, dtype=torch.uint8, device=dev))
            ob = M.DPObserver.for_env(env)
            if mode == "fused":
                env.set_observer(ob)
                fn, nbytes = (lambda e=env, o=out: e.step_into(act, *o)), base + 124
            elif mode == "two-kernel":
                ob.reset(y)

                def fn(e=env, o=out, ob=ob):
                    e.step_into(act, *o)
                    ob.step(y, thrust, angles, restart=o[2])
                    o[0][3:6].copy_(ob.nu_hat)
                fn, nbytes = fn, base + 161 + 24
            else:
                fn, nbytes = (lambda e=env, o=out: e.step_into(act, *o)), base
            runs.append(("%s%s" % (mode, tag), fn, nbytes, env, ob))
    for _, fn, _, _, _ in runs:
        for _ in range(20):
            fn()
    times = {r[0]: [] for r in runs}
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(reps):
        for name, fn, _, _, _ in runs:
            torch.cuda.synchronize()
            e0.record()
            for _ in range(steps):
                fn()
            e1.record()
            e1.synchronize()
            times[name].append(e0.elapsed_time(e1) / steps)
    rows = []
    for name, _, nbytes, _, ob in runs:
        assert torch.isfinite(ob.state).all()
        ms = float(np.median(times[name]))
        rate = n / (ms * 1e-3)
        rows.append(dict(variant=name, ms_per_step=ms, spread_ms=[float(min(times[name])), float(max(times[name]))],
                         g_env_steps_per_s=rate / 1e9, bytes_per_env_step=nbytes, hbm_fraction=rate * nbytes / (HBM_GBS * 1e9)))
    return rows


def epoch_times(dev, reps):
    rows = []
    for n in (4, 16384):
        for attached in (False, True):
            env = make_env(dev, n, True, seed=0, auto_reset=True)
            env.reset()
            if attached:
                env.set_observer(M.DPObserver.for_env(env))
            ac = M.ActorCritic(9, 7, (80, 80, 80), "leaky_relu", device=dev, seed=0)
            M.ppo(env, ac=ac, steps_per_epoch=400, epochs=3, seed=0, graph=True)           # capture
            torch.cuda.synchronize()
            t = []
            for r in range(reps):
                t0 = time.perf_counter()
                M.ppo(env, ac=ac, steps_per_epoch=400, epochs=5, seed=0, graph=True)
                torch.cuda.synchronize()
                t.append((time.perf_counter() - t0) / 5)
            rows.append(dict(n=n, observer=attached, s_per_epoch=float(np.median(t)), spread=[float(min(t)), float(max(t))]))
            print("| %d x 400 | %s | %.4f s (%.4f-%.4f) |" % (n, "attached" if attached else "none", rows[-1]["s_per_epoch"],
                                                           min(t), max(t)), flush=True)
    return rows


def hypothesis(dev, epochs, seeds, eval_steps):
    res = {"train": [], "eval": []}
    policies = {}
    for arm in ("A", "B"):
        for s in range(seeds):
            env = make_env(dev, 4, True, seed=100 + s, auto_reset=True)
            env.reset()
            if arm == "B":
                env.set_observer(M.DPObserver.for_env(env, peak_frequency=1.5))
            t0 = time.perf_counter()
            ac, hist = M.ppo(env, steps_per_epoch=400, epochs=epochs, seed=s, graph=True, hidden_sizes=(80, 80, 80),
                             activation="leaky_relu")
            last = hist[-10:]
            row = dict(arm=arm, seed=s, seconds=time.perf_counter() - t0,
                       step_reward=float(np.mean([h["AverageStepReward"] for h in last])),
                       vvals=float(np.mean([h["AverageVVals"] for h in last])),
                       eplen=float(np.mean([h["EpLen"] for h in last if h["Episodes"] > 0] or [0])),
                       at200=dict(step_reward=float(np.mean([h["AverageStepReward"] for h in hist[190:200]])),
                                  vvals=float(np.mean([h["AverageVVals"] for h in hist[190:200]])),
                                  eplen=float(np.mean([h["EpLen"] for h in hist[190:200] if h["Episodes"] > 0] or [0]))))
            res["train"].append(row)
            print("train", json.dumps(row), flush=True)
            policies[(arm, s)] = ac
    n = 6 * WE.SEEDS
    for sp in WE.SIGMAS:
        for arm in ("A", "B"):
            m_all, pos_all, yaw_all = [], [], []
            for s in range(seeds):
                env = M.RevoltFinal(M.StandInHull(), testing=True, extended_state=True, cont_ang=True, num_envs=n, device=dev,
                                    max_ep_len=2 * eval_steps, seed=11)
                if sp > 0:
                    env.set_waves(**WE.sea(sp))
                rec = evaluate.run_RL_policy(env, policies[(arm, s)], max_ep_len=eval_steps,
                                             observer=M.DPObserver.for_env(env, peak_frequency=1.5))
                eta = rec["eta"].cpu().numpy()[-100:]                    # the last 20 s
                m_all.append(rec["metrics"].cpu().numpy())
                pos_all.append(np.hypot(eta[:, 0], eta[:, 1]).mean(axis=0))
                yaw_all.append(np.rad2deg(np.abs(eta[:, 2])).mean(axis=0))
            m = np.concatenate(m_all, axis=1)
            row = dict(sigma_pos=sp, arm=arm, IAE=float(m[0].mean()), W=float(m[1].mean()), IADC=float(m[2].mean()),
                       pos_err_m=float(np.concatenate(pos_all).mean()), yaw_err_deg=float(np.concatenate(yaw_all).mean()),
                       per_seed_pos=[float(p.mean()) for p in pos_all])
            res["eval"].append(row)
            print("| %.2f | %s | %.2f | %.1f | %.3f | %.3f | %.3f |" % (sp, arm, row["IAE"], row["W"], row["IADC"],
                                                                     row["pos_err_m"], row["yaw_err_deg"]), flush=True)
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--n", type=int, default=1 << 24)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--epochs", type=int, default=800)
    ap.add_argument("--seeds", type=int, default=3)
    ap.add_argument("--eval-steps", type=int, default=400)
    ap.add_argument("--skip", default="", help="comma-separated parts to skip: a, c, d")
    ap.add_argument("--bench-parent", default=None, help="(b): a built tree of the parent commit to run bench.py against")
    ap.add_argument("--bench-runs", type=int, default=3)
    ap.add_argument("--out", default=None, help="JSON file for the raw numbers")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("observer_loop_eval.py needs a CUDA device")
    skip = set(args.skip.split(","))
    dev = torch.device("cuda", 0)
    res = {"gpu": WE.gpu_line()}
    print("GPU, power limit:", res["gpu"], flush=True)

    def save():
        if args.out:
            os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
            with open(args.out, "w") as fh:
                json.dump(res, fh, indent=1)
    if "a" not in skip:
        res["throughput"] = throughput(dev, args.n, args.steps, args.reps)
        print("(a) %d envs, %d steps per window, median (range) of %d alternating windows" % (args.n, args.steps, args.reps))
        print("| variant | ms / step | G env-steps/s | B / env-step | of %.1f GB/s |\n|---|---|---|---|---|" % HBM_GBS)
        for r in res["throughput"]:
            print("| %s | %.4f (%.4f-%.4f) | %.2f | %d | %.1f %% |" % (r["variant"], r["ms_per_step"], r["spread_ms"][0],
                                                                     r["spread_ms"][1], r["g_env_steps_per_s"],
                                                                     r["bytes_per_env_step"], 100 * r["hbm_fraction"]), flush=True)
        save()
    if args.bench_parent:
        res["bench"] = WE.bench_ab(args.bench_parent, args.steps, args.bench_runs)
        print("(b) bench.py --gpus 1 --steps %d, alternating this tree and the parent" % args.steps)
        for key in ("this", "parent"):
            print("  %-6s %s" % (key, [r.get("value") for r in res["bench"][key]]), flush=True)
        save()
    if "c" not in skip:
        print("(c) one graph-replayed PPO epoch, 80^3, waves\n| batch | observer | s / epoch |\n|---|---|---|")
        res["epoch"] = epoch_times(dev, args.reps)
        save()
    if "d" not in skip:
        print("(d) %d epochs, %d seeds per arm\n| sigma_pos m | arm | IAE | W* | IADC | LF pos err m | LF yaw err deg |\n"
              "|---|---|---|---|---|---|---|" % (args.epochs, args.seeds))
        res["hypothesis"] = hypothesis(dev, args.epochs, args.seeds, args.eval_steps)
        save()


if __name__ == "__main__":
    main()
