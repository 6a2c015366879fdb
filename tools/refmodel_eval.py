"""DP reference model (ml4ca_refmodel_step, ml4ca_pinv_pid_ff): kernel throughput and the box-test comparison of the
controllers with raw set-point steps and with the reference model.  Writes profiles/refmodel_r3.md-style tables to stdout
and the raw numbers as JSON (--out).

  (a) throughput: 16 Mi envs, 200 back-to-back launches per timed window, CUDA events, 5 windows each, timed alternately:
      refmodel_step_kernel at step_dt 0.2 s (20 sub-steps), and pinv_pid_kernel without and with feed-forward (two envs
      per thread).  Working sets far larger than L2 (1.4 GB for the reference model).  Algorithmic bytes: 84 per
      reference-model step, 80 / 92 per PID step, over 6456.5 GB/s.
  (b) box test (evaluate.box_test_schedule(), 1800 steps of 0.2 s): the shipped 80^3 policy with and without the
      deployment node's integrator, PID + QP and PID + pseudoinverse, each with raw set-point steps and with the
      reference model (the PID then with velocity feed-forward).  Calm water (every env identical), and waves
      sigma = (0.1 m, 0.1 m, 2 deg), peak frequency U(1, 2) rad/s, with the DP observer, one wave seed per env.
      IAE, W*, IADC; per leg the largest overshoot past the set-point along the leg's move; for QP the fraction of steps
      on which the +-[4, 2, 2] demand clip binds.
  (c) --bench-parent DIR: bench.py --gpus 1 --steps 200 of this tree and of the built tree DIR, alternately.
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
REF_BYTES, PID_BYTES, PID_FF_BYTES = 84, 80, 92


def throughput(dev, n, steps, reps):
    import ctypes
    from ml4ca_b200 import _lib
    g = torch.Generator(device=dev)
    g.manual_seed(0)
    L = _lib.lib()
    cfg = _lib.RefModelCfg()
    _lib.check(L.ml4ca_refmodel_cfg_default(ctypes.byref(cfg)))
    st, sp = torch.zeros(9, n, device=dev), torch.zeros(3, n, device=dev)
    sp.uniform_(-20, 20, generator=g)

    def ref_step():
        _lib.check(L.ml4ca_refmodel_step(ctypes.byref(cfg), n, _lib.ptr(sp), _lib.ptr(st), _lib.current_stream()))
    eta = torch.rand(3, n, device=dev, generator=g) * 8 - 4
    nu = torch.rand(3, n, device=dev, generator=g) * 0.6 - 0.3
    ref = torch.rand(3, n, device=dev, generator=g) * 8 - 4
    vd = torch.rand(3, n, device=dev, generator=g) * 0.2 - 0.1
    integ, tau = torch.zeros(3, n, device=dev), torch.empty(3, n, device=dev)
    n_pct, alpha = torch.empty(3, n, device=dev), torch.empty(2, n, device=dev)

    def pid(ff):
        if ff:
            return lambda: L.ml4ca_pinv_pid_ff(n, _lib.ptr(eta), _lib.ptr(nu), _lib.ptr(ref), _lib.ptr(vd), _lib.ptr(integ),
                                               None, _lib.ptr(n_pct), _lib.ptr(alpha), _lib.current_stream())
        return lambda: L.ml4ca_pinv_pid(n, _lib.ptr(eta), _lib.ptr(nu), _lib.ptr(ref), _lib.ptr(integ), None, _lib.ptr(n_pct),
                                        _lib.ptr(alpha), _lib.current_stream())
    runs = [("refmodel_step_kernel", ref_step, REF_BYTES),
            ("pinv_pid_kernel<2, false>", pid(False), PID_BYTES),
            ("pinv_pid_kernel<2, true> (feed-forward)", pid(True), PID_FF_BYTES)]
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
    assert torch.isfinite(st).all()
    rows = []
    for name, _, nbytes in runs:
        ms = float(np.median(times[name]))
        rate = n / (ms * 1e-3)
        rows.append(dict(kernel=name, ms_per_step=ms, spread_ms=[float(min(times[name])), float(max(times[name]))],
                         g_steps_per_s=rate / 1e9, bytes_per_env_step=nbytes, hbm_fraction=rate * nbytes / (HBM_GBS * 1e9),
                         hbm_floor_ms=n * nbytes / (HBM_GBS * 1e9) * 1e3))
    return rows


def overshoot(rec, steps):
    """Per leg (set-point k held from steps[k] to steps[k+1]): the largest excursion past the set-point along the leg's move,
    max over envs: m for N and E, deg for heading.  -> [legs, 3]."""
    eta, sp = rec["eta"].double().cpu().numpy(), rec["setpoint"].double().cpu().numpy()
    out = []
    for k in range(1, len(steps) - 1):
        a, b = int(steps[k]), int(steps[k + 1])
        move = sp[a] - sp[a - 1]
        e = eta[a:b + 1] - sp[a][None]
        e[:, 2] = np.rad2deg(np.mod(e[:, 2] + np.pi, 2 * np.pi) - np.pi)
        over = (np.sign(move)[None] * e).max(axis=0).clip(min=0)                      # [3, n]
        over[move == 0] = 0.0
        out.append(over.max(axis=1))
    return np.array(out)


def box_test(dev, ac, n_waves):
    steps, sp = evaluate.box_test_schedule()
    T = int(steps[-1])
    rows = []
    controllers = [("RL 80^3", "rl", False), ("RLintegral 80^3", "rl", True), ("PID + QP", "qp", None),
                   ("PID + pinv", "pinv", None)]
    for sea in ("calm", "waves"):
        n = 4 if sea == "calm" else n_waves
        for label, kind, integ in controllers:
            for with_model in (False, True):
                env = M.RevoltFinal(M.StandInHull(), testing=True, extended_state=True, cont_ang=True, num_envs=n, device=dev,
                                    max_ep_len=4 * T, seed=21)
                obs = None
                if sea == "waves":
                    env.set_waves(sigma=(0.1, 0.1, np.deg2rad(2.0)), peak_frequency=(1.0, 2.0), damping=0.1)
                    obs = M.DPObserver.for_env(env)
                model = M.ReferenceModel.for_env(env) if with_model else None
                t0 = time.perf_counter()
                if kind == "rl":
                    rec = evaluate.run_RL_policy(env, ac, integrator=integ, observer=obs, schedule=(steps, sp),
                                                 reference_model=model)
                else:
                    rec = evaluate.run_allocator(env, kind, observer=obs, schedule=(steps, sp), reference_model=model)
                m = rec["metrics"].double().cpu().numpy()
                row = dict(sea=sea, controller=label, reference_model=with_model, n=n, T=T,
                           iae=[float(m[0].mean()), float(m[0].std())], work=[float(m[1].mean()), float(m[1].std())],
                           iadc=[float(m[2].mean()), float(m[2].std())], overshoot=overshoot(rec, steps).tolist(),
                           seconds=time.perf_counter() - t0)
                if "demand_clipped" in rec:
                    row["clip_binds"] = float(rec["demand_clipped"].float().mean())
                rows.append(row)
                ov = np.array(row["overshoot"])
                print("| %s | %s | %s | %.1f +- %.1f | %.0f +- %.0f | %.1f +- %.1f | %s | %s | %s |" % (
                    sea, label, "yes" if with_model else "raw steps", row["iae"][0], row["iae"][1], row["work"][0],
                    row["work"][1], row["iadc"][0], row["iadc"][1],
                    " / ".join("%.2f" % ov[k, d] for k, d in ((0, 0), (1, 1), (3, 0))), "%.1f" % ov[2, 2],
                    "%.1f %%" % (100 * row["clip_binds"]) if "clip_binds" in row else "-"), flush=True)
    return rows


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--n", type=int, default=1 << 24)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--wave-seeds", type=int, default=48)
    ap.add_argument("--skip-throughput", action="store_true")
    ap.add_argument("--skip-box-test", action="store_true")
    ap.add_argument("--bench-parent", default=None, help="(c): a built tree of the parent commit to run bench.py against")
    ap.add_argument("--bench-runs", type=int, default=3)
    ap.add_argument("--out", default=None, help="JSON file for the raw numbers")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("refmodel_eval.py needs a CUDA device")
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
    if not args.skip_box_test:
        params = np.load(os.path.join(ROOT, "tests", "golden", "policy_final_80x3.npz"))["params"]
        ac = M.ActorCritic(9, 7, (80, 80, 80), "leaky_relu", params=params, device=dev)
        print("(b) box test, 1800 steps; calm: 4 identical envs, waves: %d seeds (mean +- std over envs)" % args.wave_seeds)
        print("| sea | controller | reference model | IAE | W* | IADC | overshoot surge / sway / combined N, m | "
              "overshoot yaw, deg | QP demand clip binds |\n|---|---|---|---|---|---|---|---|---|")
        res["box_test"] = box_test(dev, ac, args.wave_seeds)
    if args.bench_parent:
        res["bench"] = WE.bench_ab(args.bench_parent, args.steps, args.bench_runs)
        print("(c) bench.py --gpus 1 --steps %d, alternating this tree and the parent" % args.steps)
        for key in ("this", "parent"):
            print("  %-6s %s" % (key, json.dumps(res["bench"][key])), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()
