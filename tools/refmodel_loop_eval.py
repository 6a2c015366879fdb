"""DP reference model in the loop (ml4ca_env_set_refmodel, the REF variants of the env-step kernel): step time, the
headline benchmark against the parent, and whether training with the model in the loop helps the box test.  Writes
profiles/refmodel_loop_r3.md-style tables to stdout and the raw numbers as JSON (--out).

  (a) step time: 16 Mi RevoltFinal envs (extended, continuous angles), auto_reset, 200 launches per timed window, CUDA
      events, 5 windows per arm, timed alternately: the plain step; ml4ca_refmodel_step on the set-point rows, the
      set_ref copy of eta_d and the plain step; the fused REF step.  Without and with an attached observer.  Algorithmic
      bytes per env-step: 177 / 285 / 249 (301 / 409 / 373 with the observer; the separate arm adds the model's 84 B and
      the 24 B copy), over 6456.5 GB/s.
  (b) --bench-parent DIR: bench.py --gpus 1 --steps 200 of this tree and of the built tree DIR, alternately.
  (c) PPO at the reference configuration (80^3 leaky-ReLU, RevoltFinal extended with continuous angles, 4 envs x 400
      steps, graph-replayed), calm water, --epochs epochs, --seeds seeds per arm: arm A without, arm B with the model
      attached during training.  Each policy, and the shipped policy_final_80x3, is evaluated (i) on box_test_schedule()
      with the reference model (run_RL_policy(schedule=, reference_model=)) and (ii) on the 6 fixed test poses with a
      zero set-point for 400 steps (station keeping, no model): IAE against the set-point, W*, IADC, overshoot per leg.
"""
import argparse
import ctypes
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
import refmodel_eval as RE
import wave_eval as WE
from ml4ca_b200 import _lib, evaluate

HBM_GBS = WE.HBM_GBS
BYTES = {False: (177, 285, 249), True: (301, 409, 373)}     # plain, separate, fused; [observer]


def step_time(dev, n, steps, reps):
    L = _lib.lib()
    rows = []
    for obsv in (False, True):
        envs = [M.RevoltFinal(M.StandInHull(), extended_state=True, cont_ang=True, num_envs=n, device=dev, seed=s,
                              auto_reset=True) for s in (1, 2)]
        sp = torch.rand(3, n, device=dev) * 6 - 3
        for e in envs:
            e.reset()
            e.set_ref(sp)
            if obsv:
                e.set_observer(M.DPObserver.for_env(e))
        plain, fused = envs
        sep = M.ReferenceModel.for_env(plain)
        sep.reset(plain.get_state()["eta"])
        fused.set_reference_model(M.ReferenceModel.for_env(fused))
        act = torch.rand(7, n, device=dev) * 2 - 1
        obs, rew, done = torch.empty(9, n, device=dev), torch.empty(n, device=dev), torch.empty(n, dtype=torch.uint8, device=dev)
        s = _lib.current_stream()

        def separate():
            _lib.check(L.ml4ca_refmodel_step(ctypes.byref(sep.cfg), n, _lib.ptr(sp), _lib.ptr(sep.state), s))
            _lib.check(L.ml4ca_env_set_ref(plain._handle, _lib.ptr(sep.state), s))     # rows 0-2 of the state: eta_d
            plain.step_into(act, obs, rew, done)
        arms = [("step", lambda: plain.step_into(act, obs, rew, done)),
                ("refmodel_step + set_ref + step", separate),
                ("fused REF step", lambda: fused.step_into(act, obs, rew, done))]
        for _, fn in arms:
            for _ in range(20):
                fn()
        times = {name: [] for name, _ in arms}
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        for _ in range(reps):
            for name, fn in arms:
                torch.cuda.synchronize()
                e0.record()
                for _ in range(steps):
                    fn()
                e1.record()
                e1.synchronize()
                times[name].append(e0.elapsed_time(e1) / steps)
        for (name, _), nbytes in zip(arms, BYTES[obsv]):
            ms = float(np.median(times[name]))
            rows.append(dict(observer=obsv, arm=name, ms_per_step=ms, spread_ms=[float(min(times[name])), float(max(times[name]))],
                             bytes_per_env_step=nbytes, hbm_fraction=n * nbytes / (ms * 1e-3) / (HBM_GBS * 1e9)))
        del envs, plain, fused, sep
        torch.cuda.empty_cache()
    return rows


def evaluate_policy(dev, ac):
    """(i) the box test with the reference model, (ii) fixed-pose station keeping: -> dict of metrics."""
    steps, sp = evaluate.box_test_schedule()
    env = M.RevoltFinal(M.StandInHull(), testing=True, extended_state=True, cont_ang=True, num_envs=4, device=dev,
                        max_ep_len=4 * int(steps[-1]), seed=21)
    rec = evaluate.run_RL_policy(env, ac, schedule=(steps, sp), reference_model=M.ReferenceModel.for_env(env))
    m = rec["metrics"].double().cpu().numpy()
    box = dict(iae=float(m[0].mean()), work=float(m[1].mean()), iadc=float(m[2].mean()),
               overshoot=RE.overshoot(rec, steps).tolist())
    env = M.RevoltFinal(M.StandInHull(), testing=True, extended_state=True, cont_ang=True, num_envs=6, device=dev,
                        max_ep_len=400, seed=21)
    rec = evaluate.run_RL_policy(env, ac, max_ep_len=400)
    m = rec["metrics"].double().cpu().numpy()
    tail = rec["eta"].double().cpu().numpy()[-100:]                                 # the last 20 s
    sk = dict(iae=float(m[0].mean()), work=float(m[1].mean()), iadc=float(m[2].mean()),
              pos_m=float(np.hypot(tail[:, 0], tail[:, 1]).mean()), yaw_deg=float(np.rad2deg(np.abs(tail[:, 2])).mean()))
    return dict(box=box, station=sk)


def training(dev, epochs, seeds):
    rows = []
    params = np.load(os.path.join(ROOT, "tests", "golden", "policy_final_80x3.npz"))["params"]
    shipped = M.ActorCritic(9, 7, (80, 80, 80), "leaky_relu", params=params, device=dev)
    rows.append(dict(arm="shipped policy_final_80x3", seed=None, **evaluate_policy(dev, shipped)))
    for arm in ("A: without the model", "B: model attached"):
        for s in range(seeds):
            env = M.RevoltFinal(M.StandInHull(), extended_state=True, cont_ang=True, num_envs=4, device=dev, seed=s,
                                auto_reset=True)
            env.reset()
            if arm.startswith("B"):
                env.set_reference_model(M.ReferenceModel.for_env(env))
            t0 = time.perf_counter()
            ac, hist = M.ppo(env, steps_per_epoch=400, epochs=epochs, seed=s, graph=True, hidden_sizes=(80, 80, 80),
                             activation="leaky_relu")
            last = hist[-10:]
            row = dict(arm=arm, seed=s, seconds=time.perf_counter() - t0,
                       train_reward=float(np.mean([h["AverageStepReward"] for h in last])),
                       train_vvals=float(np.mean([h["AverageVVals"] for h in last])),
                       train_eplen=float(np.mean([h["EpLen"] for h in last if h["Episodes"] > 0] or [float("nan")])))
            row.update(evaluate_policy(dev, ac))
            rows.append(row)
            print(json.dumps(row), flush=True)
    return rows


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--n", type=int, default=1 << 24)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--epochs", type=int, default=800)
    ap.add_argument("--seeds", type=int, default=3)
    ap.add_argument("--skip-step-time", action="store_true")
    ap.add_argument("--skip-training", action="store_true")
    ap.add_argument("--bench-parent", default=None, help="(b): a built tree of the parent commit to run bench.py against")
    ap.add_argument("--bench-runs", type=int, default=3)
    ap.add_argument("--out", default=None, help="JSON file for the raw numbers")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("refmodel_loop_eval.py needs a CUDA device")
    dev = torch.device("cuda", 0)
    res = {"gpu": WE.gpu_line()}
    print("GPU, power limit:", res["gpu"], flush=True)
    if not args.skip_step_time:
        res["step_time"] = step_time(dev, args.n, args.steps, args.reps)
        print("(a) %d envs, %d launches per window, median (range) of %d alternating windows" % (args.n, args.steps, args.reps))
        print("| observer | arm | ms / step | B / env-step | of 6456.5 GB/s |\n|---|---|---|---|---|")
        for r in res["step_time"]:
            print("| %s | %s | %.4f (%.4f-%.4f) | %d | %.1f %% |" % ("yes" if r["observer"] else "no", r["arm"], r["ms_per_step"],
                  r["spread_ms"][0], r["spread_ms"][1], r["bytes_per_env_step"], 100 * r["hbm_fraction"]), flush=True)
    if args.bench_parent:
        res["bench"] = WE.bench_ab(args.bench_parent, args.steps, args.bench_runs)
        print("(b) bench.py --gpus 1 --steps %d, alternating this tree and the parent" % args.steps)
        for key in ("this", "parent"):
            print("  %-6s %s" % (key, json.dumps(res["bench"][key])), flush=True)
    if not args.skip_training:
        print("(c) PPO 80^3, 4 x 400, %d epochs, calm water" % args.epochs, flush=True)
        res["training"] = training(dev, args.epochs, args.seeds)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()
