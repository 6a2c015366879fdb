"""Batched PPO pieces mirroring /root/reference/src/rl/windows_workspace/spinup/algos/tf1/ppo/ppo.py.

  TrajectoryBuffer  ppo.py:21-105   device-resident [T, ., n_env] buffers, GAE-lambda by one kernel launch
  rollout()         ppo.py:289-322  T steps of (policy forward -> env step) for every environment at once

Everything heavy runs behind the C ABI (csrc/policy.cu, csrc/env_step*.cu, csrc/gae.cu); this module is plumbing.
"""

import torch

from . import _lib


class TrajectoryBuffer(object):
    """ppo.py:21-105 for n_env environments x T steps, on the device.

    Layout [T, component, n_env] (time-major, struct-of-arrays inside a step) so that each rollout
    step writes contiguous rows.  ``val`` has T + 1 rows: row T holds the bootstrap values V(s_T)
    (ppo.py:311)."""

    def __init__(self, obs_dim, act_dim, size, num_envs, gamma=0.99, lam=0.95, device=None, max_ep_len=None):
        self.device = torch.device(device if device is not None else "cuda")
        T, n = int(size), int(num_envs)
        # ppo.py:303-311 inside the buffer: `last_val = v(o)` at an episode-length cut.  Two cuts of one env are at least
        # max_ep_len steps apart, so one bootstrap row per window of (at most) max_ep_len steps is enough (ml4ca_gae,
        # boot_window).  Without max_ep_len here, rollout() sizes the rows from the env it is given.
        self.boot_window = min(int(max_ep_len), T) if max_ep_len else None
        windows = (T + self.boot_window - 1) // self.boot_window if self.boot_window else 0
        f = dict(dtype=torch.float32, device=self.device)
        self._obs_rows = torch.zeros(T + 1, obs_dim, n, **f)   # row t = observation the policy acts on at step t; row T =
        self.obs_buf = self._obs_rows[:T]                      # the observation after the last step (no per-step copy)
        self.act_buf = torch.zeros(T, act_dim, n, **f)
        self.adv_buf = torch.zeros(T, n, **f)
        self.rew_buf = torch.zeros(T, n, **f)
        self.ret_buf = torch.zeros(T, n, **f)
        self.val_buf = torch.zeros(T + 1, n, **f)
        self.logp_buf = torch.zeros(T, n, **f)
        self.done_buf = torch.zeros(T, n, dtype=torch.uint8, device=self.device)
        self.cut_obs = torch.zeros(obs_dim, n, **f)            # observation returned at the cut (ml4ca_env_set_cut_obs)
        self.boot_buf = torch.zeros(windows, n, **f) if windows else None   # V(cut_obs), one row per window
        self._scratch = (torch.empty(act_dim, n, **f), torch.empty(n, **f))   # unused outputs of the bootstrap forward
        self.gamma, self.lam = gamma, lam
        self.ptr, self.max_size, self.num_envs = 0, T, n
        self._sums = torch.zeros(3, dtype=torch.float64, device=self.device)

    def finish_path(self, last_val=None, boot="buffer", boot_window=None):
        """ppo.py:65-91 for every environment at once: GAE-lambda advantages and rewards-to-go, with the path ends
        taken from the recorded done flags.  ``last_val`` [n] = V(o_T) for the epoch-end bootstrap (ppo.py:311);
        by default row T of ``val_buf`` as left by the caller.  ``boot`` = V of the observation returned at
        episode-length cuts inside the buffer: by default ``boot_buf`` as filled by rollout(); a [T, n] tensor with
        boot_window=1; None = the V(s_t) stand-in."""
        if last_val is not None:
            self.val_buf[self.max_size].copy_(last_val)
        if isinstance(boot, str):
            boot, boot_window = self.boot_buf, self.boot_window     # None before the first rollout(): V(s_t) stands in
        elif boot is not None and boot_window is None:
            boot_window = 1
        with torch.cuda.device(self.device):
            _lib.check(_lib.lib().ml4ca_gae(self.num_envs, self.max_size, _lib.ptr(self.rew_buf), _lib.ptr(self.val_buf),
                                            _lib.ptr(self.done_buf), _lib.ptr(boot), int(boot_window or 1),
                                            float(self.gamma), float(self.lam),
                                            _lib.ptr(self.adv_buf), _lib.ptr(self.ret_buf), _lib.current_stream()),
                       "ml4ca_gae")

    def get(self):
        """ppo.py:93-105: advantage normalisation with statistics over ALL ranks, then the five training arrays."""
        from . import mpi_tools
        m = self.adv_buf.numel()
        with torch.cuda.device(self.device):
            _lib.check(_lib.lib().ml4ca_stats(m, _lib.ptr(self.adv_buf), _lib.ptr(self._sums), _lib.current_stream()))
            mpi_tools.allreduce_sum_(self._sums)
            mean, std = mpi_tools.statistics_from_sums(self._sums.tolist())
            _lib.check(_lib.lib().ml4ca_normalize(m, _lib.ptr(self.adv_buf), mean, std, _lib.current_stream()))
        self.ptr = 0
        return [self.obs_buf, self.act_buf, self.adv_buf, self.ret_buf, self.logp_buf]


def _rollout_launches(env, ac, buf, seed, start_step, deterministic):
    """The 2T kernel launches of one rollout on the current stream; nothing else (capturable)."""
    L = _lib.lib()
    T, n = buf.max_size, env.num_envs
    stream = _lib.current_stream()
    W = buf.boot_window

    def bootstrap_window(t):
        # ppo.py:311 for the cuts of the window that step t closes: V of the observations the env kernels saved into
        # buf.cut_obs.  One extra forward per max_ep_len steps; columns without a cut hold stale values nobody reads.
        if (t + 1) % W == 0 or t == T - 1:
            _lib.check(L.ml4ca_policy_forward(ac._handle, n, _lib.ptr(buf.cut_obs), seed & 0xFFFFFFFFFFFFFFFF, 0, 1,
                                              env._cfg.env_id_offset, _lib.ptr(buf._scratch[0]), _lib.ptr(buf.boot_buf[t // W]),
                                              _lib.ptr(buf._scratch[1]), None, stream), "ml4ca_policy_forward")

    rows = buf._obs_rows     # row t = observation acted on at step t; the env kernel writes row t + 1 directly (no per-step copy)
    for t in range(T):
        _lib.check(L.ml4ca_policy_forward(ac._handle, n, _lib.ptr(rows[t]), seed & 0xFFFFFFFFFFFFFFFF, start_step + t,
                                          int(bool(deterministic)), env._cfg.env_id_offset, _lib.ptr(buf.act_buf[t]),
                                          _lib.ptr(buf.val_buf[t]), _lib.ptr(buf.logp_buf[t]), None, stream),
                   "ml4ca_policy_forward")
        env.step_into(buf.act_buf[t], rows[t + 1], buf.rew_buf[t], buf.done_buf[t])
        bootstrap_window(t)


def rollout(env, ac, buf, seed=0, start_step=0, deterministic=False, graph=False):
    """Fill ``buf`` with T = buf.max_size steps of every environment (ppo.py:290-302 batched).

    One policy kernel and one env-step kernel per time step; the env kernel writes the next observation row of the buffer
    directly.  (A single fused kernel was built in three arrangements and measured slower every time: profiles/rollout_r2.md.)
    graph=True: the T steps are captured once into a CUDA graph (per env / policy / buffer) and replayed on later calls --
    for small and medium batches the rollout is launch-bound (2T launches through ctypes); the Philox step number then comes
    from a device counter (ml4ca_policy_set_step_counter) that is set to ``start_step`` before every replay, so a graph
    rollout draws exactly the noise of the eager one.  The first call runs eagerly (it also initialises the kernels).
    The env must have auto_reset=True (finished episodes restart in-kernel) and must have been reset: both are checked.
    The observations returned at episode-length cuts go to ``buf.cut_obs`` and their values to ``buf.boot_buf``
    (ppo.py:311), window by window.
    Returns the observation after the last step (for the bootstrap value).
    """
    T = buf.max_size
    if not env._cfg.auto_reset:
        raise ValueError("rollout() steps every env T times without looking at `done`: the env must be created with "
                         "auto_reset=True (the reference's caller resets at ppo.py:322; here the kernel does)")
    if not getattr(env, "_has_reset", False):
        raise RuntimeError("rollout() before reset(): the env holds no observation yet")
    if buf.boot_window is None or buf.boot_window > env.max_ep_len:   # at most one cut per env and window
        buf.boot_window = min(int(env.max_ep_len), T)
        buf.boot_buf = torch.zeros((T + buf.boot_window - 1) // buf.boot_window, env.num_envs, dtype=torch.float32,
                                   device=buf.device)
        buf.__dict__.pop("_rollout_graphs", None)                     # captured graphs hold the old rows
    _lib.check(_lib.lib().ml4ca_env_set_cut_obs(env._handle, _lib.ptr(buf.cut_obs)), "ml4ca_env_set_cut_obs")
    buf._obs_rows[0].copy_(env._obs)   # observation returned by the last reset() / step()
    if not graph:
        _rollout_launches(env, ac, buf, seed, start_step, deterministic)
    else:
        cache = buf.__dict__.setdefault("_rollout_graphs", {})
        # launch parameters are baked into a captured graph: the restart fraction (curriculum), the disturbance, the
        # wave setting, the attached observer and the attached reference model are part of the key
        obsv = getattr(env, "_observer", None)
        obsv_key = None if obsv is None else (id(obsv), obsv.state.data_ptr(), obsv.omega_o.data_ptr(),
                                              bytes(obsv.cfg))
        refm = getattr(env, "_refmodel", None)
        ref_key = None if refm is None else (id(refm), refm.state.data_ptr(), bytes(refm.cfg))
        key = (id(env), id(ac), int(seed), bool(deterministic), float(env._cfg.reset_fraction),
               getattr(env, "_disturbance", None), getattr(env, "_waves", None), obsv_key, ref_key)
        entry = cache.get(key)
        if entry is None:                  # first call: eager, and remember that the next one may capture
            cache[key] = {"graph": None, "counter": torch.zeros(1, dtype=torch.int32, device=buf.device)}
            _rollout_launches(env, ac, buf, seed, start_step, deterministic)
        else:
            L = _lib.lib()
            if entry["graph"] is None:
                _lib.check(L.ml4ca_policy_set_step_counter(ac._handle, _lib.ptr(entry["counter"])))
                try:
                    torch.cuda.synchronize(buf.device)
                    g = torch.cuda.CUDAGraph()
                    with torch.cuda.graph(g, capture_error_mode="relaxed"):
                        _rollout_launches(env, ac, buf, seed, 0, deterministic)     # step = counter + t
                finally:
                    _lib.check(L.ml4ca_policy_set_step_counter(ac._handle, None))
                entry["graph"] = g
            v = int(start_step) & 0xFFFFFFFF                       # the kernel adds it as uint32
            entry["counter"].fill_(v - (1 << 32) if v >= (1 << 31) else v)
            entry["graph"].replay()
    _lib.check(_lib.lib().ml4ca_env_set_cut_obs(env._handle, None))   # the launches (or the graph) hold the pointer
    env._obs = buf._obs_rows[T].clone()
    return env._obs


class PPOUpdater(object):
    """The update() closure of ppo.py:260-280 for a device-resident buffer: full-batch gradient of pi_loss / v_loss by
    one kernel launch each (ml4ca_ppo_grad), ONE all-reduce of the flat gradient with the loss statistics in its tail
    (MpiAdamOptimizer.compute_gradients, mpi_tf.py:59-62), TF-1 Adam on the flat master parameters (ml4ca_adam_step),
    early stopping of the policy iterations on the rank-averaged approx-KL (ppo.py:268-271)."""

    def __init__(self, ac, clip_ratio=0.2, pi_lr=3e-4, vf_lr=1e-3, train_pi_iters=80, train_v_iters=80, target_kl=0.01):
        self.ac = ac
        self.clip_ratio, self.pi_lr, self.vf_lr = float(clip_ratio), float(pi_lr), float(vf_lr)
        self.train_pi_iters, self.train_v_iters, self.target_kl = int(train_pi_iters), int(train_v_iters), float(target_kl)
        dev, P = ac.device, ac.num_params
        self.n_pi = ac.var_counts[0]                 # pi variables + log_std come first in the flat vector
        self.flat = torch.zeros(P + 8, dtype=torch.float32, device=dev)      # gradient | 5 statistics (+ pad)
        self.stats = torch.zeros(8, dtype=torch.float64, device=dev)
        self.m1 = torch.zeros(P, dtype=torch.float32, device=dev)
        self.m2 = torch.zeros(P, dtype=torch.float32, device=dev)
        self.t_pi = self.t_v = 0
        # policy loop: two (gradient, statistics) slots so that the pass of iteration i + 1 can be queued while the host is still
        # waiting for the KL of iteration i (update())
        self._flat2 = torch.zeros(P + 8, dtype=torch.float32, device=dev)
        self._stats2 = torch.zeros(8, dtype=torch.float64, device=dev)
        self._host = [torch.zeros(5, dtype=torch.float32).pin_memory() for _ in range(2)]
        self._events = [torch.cuda.Event() for _ in range(2)]
        # ranks = GPUs of one node: the all-reduce of the flat gradient runs over NVLink peer memory inside the kernel that
        # applies the Adam step (csrc/peer_comm.cu); None = single rank or peers not mappable -> NCCL all-reduce
        from . import mpi_tools
        self.peer = mpi_tools.PeerComm.create(P + 8, dev)

    # -- one gradient pass: returns the rank-summed statistics as a list of 5 floats and the global sample count ------
    def _slot(self, slot):
        return (self.flat, self.stats) if slot == 0 else (self._flat2, self._stats2)

    def _grad(self, net, data, T, n, read=True, slot=0):
        """One gradient pass.  read=False leaves the statistics on the device (no host synchronisation): (None, count).
        read='async': the five statistics are copied to a pinned host slot behind the pass and an event is recorded;
        ``_read(slot)`` later waits for that event only, not for work queued after it."""
        obs, act, adv, ret, logp = data
        L, ac = _lib.lib(), self.ac
        flat, stats = self._slot(slot)
        with torch.cuda.device(ac.device):
            _lib.check(L.ml4ca_ppo_grad(ac._handle, int(net), int(n), int(T), _lib.ptr(obs), _lib.ptr(act), _lib.ptr(adv),
                                        _lib.ptr(ret), _lib.ptr(logp), self.clip_ratio, _lib.ptr(flat),
                                        _lib.ptr(stats), _lib.current_stream()), "ml4ca_ppo_grad")
        from . import mpi_tools
        P = ac.num_params
        self._exchange(flat, stats)
        count = float(T) * float(n) * mpi_tools.num_procs()   # equal shards (mpi_tools.shard_bounds differ by <= 1 env)
        if read == 'async':
            self._host[slot].copy_(flat[P:P + 5], non_blocking=True)
            self._events[slot].record()
            return None, count
        return (flat[P:P + 5].tolist() if read else None), count

    def _exchange(self, flat, stats, ctl=None, it=0):
        """Sum of the flat gradient (+ the five statistics, moved into its tail) over the ranks, in place."""
        from . import mpi_tools
        P = self.ac.num_params
        if self.peer is not None:
            with torch.cuda.device(self.ac.device):
                _lib.check(_lib.lib().ml4ca_peer_allreduce(self.peer._handle, _lib.ptr(flat), P + 8, _lib.ptr(stats), P, 5,
                                                           None if ctl is None else _lib.ptr(ctl), int(it), _lib.current_stream()),
                           "ml4ca_peer_allreduce")
        else:
            flat[P:P + 5].copy_(stats[:5])
            mpi_tools.allreduce_sum_(flat)

    def _read(self, slot):
        self._events[slot].synchronize()
        return self._host[slot].tolist()

    def _adam(self, net, count, slot=0):
        ac, L = self.ac, _lib.lib()
        flat = self._slot(slot)[0]
        lo, hi = (0, self.n_pi) if net == 0 else (self.n_pi, ac.num_params)
        if net == 0:
            self.t_pi += 1
        else:
            self.t_v += 1
        t, lr = (self.t_pi, self.pi_lr) if net == 0 else (self.t_v, self.vf_lr)
        params = ac.parameters()
        with torch.cuda.device(ac.device):
            _lib.check(L.ml4ca_adam_step(hi - lo, _lib.ptr(params[lo:hi]), _lib.ptr(flat[lo:hi]), _lib.ptr(self.m1[lo:hi]),
                                         _lib.ptr(self.m2[lo:hi]), lr, 0.9, 0.999, 1e-8, t, 1.0 / count,
                                         _lib.current_stream()), "ml4ca_adam_step")
        # the fp16 operand image of the forward kernel is NOT refreshed here: the gradient kernels read the fp32 master
        # parameters, so update() refreshes it once, after the last step

    def losses(self, data, T, n):
        """pi_loss, v_loss, approx_kl, approx_ent, clipfrac at the current parameters (ppo.py:262,275)."""
        s, c = self._grad(0, data, T, n)
        out = {"LossPi": -s[0] / c, "KL": s[2] / c, "Entropy": s[3] / c, "ClipFrac": s[4] / c}
        s, c = self._grad(1, data, T, n)
        out["LossV"] = s[1] / c
        return out

    def _update_v(self, data, T, n, info):
        """ppo.py:272-273 / trpo.py:323-325: train_v_iters Adam steps on v_loss."""
        for i in range(self.train_v_iters):      # nothing to test between the steps: only the first pass is read back
            s, c = self._grad(1, data, T, n, read=(i == 0))
            if i == 0:
                info["LossV"] = s[1] / c
            self._adam(1, c)

    # -- the whole update as one CUDA graph ------------------------------------------------------------------------------
    def _capture_update(self, data, T, n):
        """Capture [ctl_begin | pi loop | v loop | ctl_end | refresh | the two loss passes] into one CUDA graph.  The early
        stop of the policy loop lives on the device (ml4ca_ppo_ctl): the passes of the iterations behind the stopping one
        return at once, so the host neither launches per iteration nor waits for a KL.  Returns (graph, ctl, out)."""
        from . import mpi_tools
        ac, L = self.ac, _lib.lib()
        dev, P = ac.device, ac.num_params
        obs, act, adv, ret, logp = data
        ctl = getattr(self, "_ctl", None)
        if ctl is None:
            ctl = self._ctl = torch.zeros(12, dtype=torch.int32, device=dev)       # struct ml4ca_ppo_ctl
            ctl[2], ctl[3] = self.t_pi, self.t_v
        out = torch.zeros(16, dtype=torch.float32, device=dev)                      # statistics of the closing loss passes
        count = float(T) * float(n) * mpi_tools.num_procs()
        flat, stats, params = self.flat, self.stats, ac.parameters()
        kl_limit = 1.5 * self.target_kl

        def one_pass(net, it, use_ctl, exchange=True):
            _lib.check(L.ml4ca_ppo_grad_ex(ac._handle, net, int(n), int(T), _lib.ptr(obs), _lib.ptr(act), _lib.ptr(adv), _lib.ptr(ret),
                                           _lib.ptr(logp), self.clip_ratio, _lib.ptr(flat), _lib.ptr(stats),
                                           _lib.ptr(ctl) if use_ctl else None, it, _lib.current_stream()), "ml4ca_ppo_grad_ex")
            if exchange:
                self._exchange(flat, stats, ctl if use_ctl else None, it)

        def launches():
            st = _lib.current_stream()
            _lib.check(L.ml4ca_ppo_ctl_begin(_lib.ptr(ctl), st))
            for net, iters, lr, limit in ((0, self.train_pi_iters, self.pi_lr, kl_limit), (1, self.train_v_iters, self.vf_lr, 0.0)):
                lo, hi = (0, self.n_pi) if net == 0 else (self.n_pi, P)
                for it in range(iters):
                    if self.peer is not None:      # exchange + Adam + early-stop test in one kernel over NVLink peer memory
                        one_pass(net, it, net == 0, exchange=False)
                        _lib.check(L.ml4ca_adam_step_peer(self.peer._handle, _lib.ptr(flat), P + 8, _lib.ptr(stats), P, lo, hi,
                                                          _lib.ptr(params), _lib.ptr(self.m1), _lib.ptr(self.m2), lr, 0.9, 0.999, 1e-8,
                                                          1.0 / count, net, it, count, limit, _lib.ptr(ctl), st), "ml4ca_adam_step_peer")
                        continue
                    one_pass(net, it, net == 0)
                    _lib.check(L.ml4ca_adam_step_dev(hi - lo, _lib.ptr(params[lo:hi]), _lib.ptr(flat[lo:hi]), _lib.ptr(self.m1[lo:hi]),
                                                     _lib.ptr(self.m2[lo:hi]), lr, 0.9, 0.999, 1e-8, 1.0 / count, net, it,
                                                     _lib.ptr(flat[P:P + 5]), count, limit, _lib.ptr(ctl), st), "ml4ca_adam_step_dev")
            _lib.check(L.ml4ca_ppo_ctl_end(_lib.ptr(ctl), self.train_pi_iters, self.train_v_iters, st))
            _lib.check(L.ml4ca_policy_refresh(ac._handle, st), "ml4ca_policy_refresh")
            one_pass(0, 0, False)
            out[0:5].copy_(flat[P:P + 5])
            one_pass(1, 0, False)
            out[5:10].copy_(flat[P:P + 5])

        with torch.cuda.device(dev):
            torch.cuda.synchronize(dev)
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, capture_error_mode="relaxed"):
                launches()
        return g, ctl, out

    def update_graph(self, buf):
        """update() replayed from one CUDA graph (captured on the first call per buffer): same arithmetic, same early stop
        (ppo.py:268-271: the step of the stopping iteration is applied), one launch and one read-back per epoch."""
        data = buf.get()
        T, n = buf.max_size, buf.num_envs
        cache = self.__dict__.setdefault("_update_graphs", {})
        key = (id(buf), T, n)
        if key not in cache:
            cache[key] = self._capture_update(data, T, n)
        g, ctl, out = cache[key]
        ctl[2], ctl[3] = self.t_pi, self.t_v        # eager updates in between advance the host-side step counts
        g.replay()
        c = float(T) * float(n) * __import__("ml4ca_b200").mpi_tools.num_procs()
        host = torch.cat([ctl.view(torch.float32).clone(), out]).cpu()             # the one read-back of the epoch
        ints = host[:4].view(torch.int32).tolist()
        first, o = host[4:12].tolist(), host[12:28].tolist()
        self.t_pi, self.t_v = ints[2], ints[3]
        info = {"StopIter": ints[1], "LossPi": -first[0] / c, "Entropy": first[3] / c, "LossV": first[5] / c,
                "KL": o[2] / c, "ClipFrac": o[4] / c}
        info["DeltaLossPi"] = -o[0] / c - info["LossPi"]
        info["DeltaLossV"] = o[6] / c - info["LossV"]
        return info

    def update(self, buf, graph=False):
        """ppo.py:260-280.  ``buf`` = a TrajectoryBuffer after finish_path(); returns the logger's dictionary.
        graph=True: the whole update from one CUDA graph with a device-side KL stop (update_graph)."""
        if graph:
            return self.update_graph(buf)
        if getattr(self, "_ctl", None) is not None:          # keep the device-side step counts in step with the host's
            self._ctl[2], self._ctl[3] = self.t_pi, self.t_v
        data = buf.get()
        T, n = buf.max_size, buf.num_envs
        info, stop = {}, 0
        # The KL of iteration i (ppo.py:268-271) is only known after a device -> host round trip; instead of idling the GPU for
        # it, the Adam step of iteration i (always applied) and the gradient pass of iteration i + 1 are queued first, into
        # the other slot.  When the test stops the loop that pass was for nothing: it changes no parameter.
        _, c = self._grad(0, data, T, n, read='async', slot=0)
        for i in range(self.train_pi_iters):
            cur = i & 1
            self._adam(0, c, slot=cur)
            if i + 1 < self.train_pi_iters:
                self._grad(0, data, T, n, read='async', slot=cur ^ 1)
            s = self._read(cur)                       # loss statistics belong to the parameters BEFORE this step
            if i == 0:
                info.update(LossPi=-s[0] / c, Entropy=s[3] / c)
            stop = i
            if s[2] / c > 1.5 * self.target_kl:       # kl = mpi_avg(kl): the step of this iteration has been applied
                break
        info["StopIter"] = stop
        self._update_v(data, T, n, info)
        self.ac.refresh()
        new = self.losses(data, T, n)
        info.update(KL=new["KL"], ClipFrac=new["ClipFrac"], DeltaLossPi=new["LossPi"] - info.get("LossPi", new["LossPi"]),
                    DeltaLossV=new["LossV"] - info.get("LossV", new["LossV"]))
        return info


class _GraphUpdater(object):
    """PPOUpdater whose update() replays the captured graph (what run_epochs calls)."""

    def __init__(self, upd):
        self.inner = upd

    def update(self, buf):
        return self.inner.update_graph(buf)


PPO_COLUMNS = ('LossPi', 'LossV', 'DeltaLossPi', 'DeltaLossV', 'Entropy', 'KL', 'ClipFrac', 'StopIter')   # ppo.py:339-346


def ppo(env, ac=None, steps_per_epoch=400, epochs=1, gamma=0.99, clip_ratio=0.2, pi_lr=3e-4, vf_lr=1e-3,
        train_pi_iters=80, train_v_iters=80, lam=0.97, target_kl=0.01, seed=0, hidden_sizes=(64, 64),
        activation="leaky_relu", logger=None, logger_kwargs=None, graph=False, curriculum=False,
        reset_each_epoch=True, update_graph=None):
    """ppo.py:107-346 for a batched env: every epoch = ``steps_per_epoch`` steps of EVERY environment of ``env``
    (rollout), GAE-lambda (finish_path), advantage normalisation over all ranks, then the PPO update.
    Hyper-parameter defaults are the reference's config.json.  ``logger_kwargs=dict(output_dir=..., exp_name=...)``
    writes progress.txt / config.json in the reference's format (ppo.py:332-346, logx.py).  ``logger`` may be a callable
    receiving each epoch's dictionary.  ``curriculum`` (ppo.py:286,319): resets sample from fraction 0 at the start,
    min(3 epoch / epochs, 0.8) afterwards.  ``reset_each_epoch`` (ppo.py:304,322: the reference also resets the env when
    the epoch ends).  Returns (ac, list of per-epoch dictionaries)."""
    from . import mpi_tools
    from .core import ActorCritic
    n, dev = env.num_envs, env.device
    if ac is None:
        ac = ActorCritic(env.num_states, env.num_actions, hidden_sizes, activation, device=dev, seed=seed)
    params = ac.parameters()
    mpi_tools.sync_all_params(params)             # ppo.py:255
    ac.refresh()
    buf = TrajectoryBuffer(env.num_states, env.num_actions, steps_per_epoch, n, gamma, lam, device=dev,
                           max_ep_len=env.max_ep_len)
    upd = PPOUpdater(ac, clip_ratio, pi_lr, vf_lr, train_pi_iters, train_v_iters, target_kl)
    if update_graph if update_graph is not None else graph:    # graph=True also replays the update from a CUDA graph
        upd = _GraphUpdater(upd)
    config = dict(steps_per_epoch=steps_per_epoch, epochs=epochs, gamma=gamma, clip_ratio=clip_ratio, pi_lr=pi_lr,
                  vf_lr=vf_lr, train_pi_iters=train_pi_iters, train_v_iters=train_v_iters, lam=lam,
                  target_kl=target_kl, seed=seed)
    return run_epochs(env, ac, buf, upd, steps_per_epoch, epochs, seed, logger, logger_kwargs, config, PPO_COLUMNS,
                      log_std_column=True, graph=graph, curriculum=curriculum, reset_each_epoch=reset_each_epoch)


def run_epochs(env, ac, buf, upd, steps_per_epoch, epochs, seed, logger, logger_kwargs, config, columns,
               log_std_column=False, graph=False, curriculum=False, reset_each_epoch=True):
    """The epoch loop shared by ppo() (ppo.py:283-346) and trpo() (trpo.py:327-384): rollout of every environment,
    bootstrap + GAE-lambda (cuts inside the buffer bootstrap with V of the observation returned at the cut, the buffer
    end with V of the last observation: ppo.py:311 both), episode / value statistics, ``upd.update(buf)``, the
    reference's progress.txt columns.  With ``reset_each_epoch`` every env restarts when the epoch ends, as the
    reference's loop does (`terminal or t == local_steps_per_epoch - 1` -> env.reset, ppo.py:304,322)."""
    import time as _time
    from . import logx, mpi_tools
    n, dev = env.num_envs, env.device
    flog = None
    if logger_kwargs is not None:
        flog = logx.Logger(rank=mpi_tools.proc_id(), **logger_kwargs)
        flog.save_config(dict(config, max_ep_len=env.max_ep_len, num_envs=n,
                              num_procs=mpi_tools.num_procs(), actor_critic="mlp_actor_critic",
                              ac_kwargs=dict(hidden_sizes=list(ac.hidden_sizes), activation=ac.activation)))
    run_ret = torch.zeros(n, dtype=torch.float32, device=dev)
    run_len = torch.zeros(n, dtype=torch.int32, device=dev)
    s5 = torch.zeros(3, 5, dtype=torch.float64, device=dev)       # EpRet, EpLen, VVals
    L = _lib.lib()
    if not env._cfg.auto_reset:
        raise ValueError("the training loop needs an env created with auto_reset=True (see rollout())")
    env.reset(fraction=0.0 if curriculum else 0.8)                    # ppo.py:286
    history, step, start_time = [], 0, _time.time()
    for epoch in range(epochs):
        fraction = min(3.0 * epoch / epochs, 0.8) if curriculum else 0.8   # ppo.py:319
        env.set_reset_fraction(fraction)                              # what the restarts inside this epoch sample with
        o_last = rollout(env, ac, buf, seed=seed, start_step=step, graph=graph)
        step += steps_per_epoch
        _, v_last, _ = ac.step(o_last, deterministic=True, step=step)
        buf.finish_path(last_val=v_last)          # ppo.py:311 for the envs still running at the epoch end
        with torch.cuda.device(dev):
            st = _lib.current_stream()
            _lib.check(L.ml4ca_episode_stats(n, steps_per_epoch, _lib.ptr(buf.rew_buf), _lib.ptr(buf.done_buf), _lib.ptr(run_ret),
                                             _lib.ptr(run_len), _lib.ptr(s5[0]), _lib.ptr(s5[1]), st), "ml4ca_episode_stats")
            _lib.check(L.ml4ca_stats5(steps_per_epoch * n, _lib.ptr(buf.val_buf), _lib.ptr(s5[2]), st), "ml4ca_stats5")
        red = s5.clone()
        mpi_tools.allreduce_sum_(red[:, 0:3])
        if mpi_tools.num_procs() > 1:
            lo, hi = red[:, 3].clone(), red[:, 4].clone()
            torch.distributed.all_reduce(lo, op=torch.distributed.ReduceOp.MIN)
            torch.distributed.all_reduce(hi, op=torch.distributed.ReduceOp.MAX)
            red[:, 3], red[:, 4] = lo, hi
        red = red.tolist()
        rew_mean = float(mpi_tools.mpi_avg(buf.rew_buf.mean().item()))
        if reset_each_epoch:                      # ppo.py:322 at t == local_steps_per_epoch - 1 (trajectory cut by the epoch)
            env.reset(fraction=fraction)
            run_ret.zero_()
            run_len.zero_()
        info = upd.update(buf)
        info.update(Epoch=epoch, AverageStepReward=rew_mean,
                    TotalEnvInteracts=(epoch + 1) * steps_per_epoch * n * mpi_tools.num_procs(),
                    AverageEpRet=logx.statistics_from5(red[0])[0], EpLen=logx.statistics_from5(red[1])[0],
                    AverageVVals=logx.statistics_from5(red[2])[0], Episodes=int(red[0][2]))
        history.append(info)
        if flog is not None:                      # the reference's columns, in its order (ppo.py:332-346)
            flog.log_tabular('Epoch', epoch)
            flog.log_stats('EpRet', red[0], with_min_and_max=True)
            flog.log_stats('EpLen', red[1], average_only=True)
            flog.log_stats('VVals', red[2], with_min_and_max=True)
            flog.log_tabular('TotalEnvInteracts', info['TotalEnvInteracts'])
            for k in columns:
                flog.log_tabular(k, info[k])
            flog.log_tabular('Time', _time.time() - start_time)
            if log_std_column:
                off = ac.var_counts[0] - ac.act_dim
                flog.log_tabular('MeanLogStd', float(ac.parameters()[off:off + ac.act_dim].mean().item()))
            flog.dump_tabular()
        if logger is not None:
            logger(info)
    return ac, history
