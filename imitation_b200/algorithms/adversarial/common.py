"""`AdversarialTrainer`: the GAIL/AIRL round on the GPU behind the reference's API.

Mirror of /root/reference/src/imitation/algorithms/adversarial/common.py: same keyword-only
constructor (:112-132), attributes (`venv`, `venv_buffering`, `venv_wrapped`, `venv_train`,
`gen_algo`, `gen_train_timesteps`, `_gen_replay_buffer`, `policy`, `reward_train`,
`reward_test`, `_global_step`, ...), methods `train` (:427-461), `train_gen` (:391-425),
`train_disc` (:317-389), `logits_expert_is_high`, `set_demonstrations` (:306-315), error
messages (:193-194, :548-562) and the 9-key stats dict of `compute_train_stats` (:27-92).

What differs is where the work happens: expert demonstrations and the generator replay ring are
HBM tables; one `train_disc` is [index sampling -> gather -> (log pi) -> RunningNorm update ->
fused forward/BCE/backward -> reduce -> Adam + stats] as ~7 launches with no host round trip
except the final 9-float read that the reference's `Mapping[str, float]` return type demands.
Additive keyword arguments: `sampling` ("device" = Philox/Feistel on the GPU, "host_compat" =
the reference's NumPy/torch RNG streams for bit-exact index parity), `seed`.
"""
import abc
import contextlib
import itertools
from typing import Callable, Mapping, Optional, Type

import numpy as np
import torch as th
from torch.nn import functional as F

from ... import _desc, _lib
from ...data import buffer, types, wrappers
from ...rewards import reward_nets, reward_wrapper
from ...util import networks
from .. import base

STAT_KEYS = ("disc_loss", "disc_acc", "disc_acc_expert", "disc_acc_gen", "disc_entropy",
             "disc_proportion_expert_true", "disc_proportion_expert_pred", "n_expert", "n_generated")


def compute_train_stats(disc_logits_expert_is_high: th.Tensor, labels_expert_is_one: th.Tensor,
                        disc_loss: th.Tensor) -> Mapping[str, float]:
    """Torch restatement of common.py:27-92 for the generic (non-fused optimiser) path; the fused
    path computes the same nine numbers inside the kernels (csrc/imb_disc.cu:write_train_stats)."""
    with th.no_grad():
        logits, labels = disc_logits_expert_is_high, labels_expert_is_one
        pred_gen, true_gen = logits < 0, labels == 0
        n_gen, n_lab = float(true_gen.sum()), float(len(labels))
        n_exp = n_lab - n_gen
        correct = pred_gen == true_gen
        n_exp_pred = n_lab - float(pred_gen.sum())
        nan = float("nan")
        ent = th.distributions.Bernoulli(logits=logits.float()).entropy().mean() if n_lab > 0 else th.tensor(nan)
        return {
            "disc_loss": float(th.mean(disc_loss)),
            "disc_acc": float(correct.float().mean()) if n_lab > 0 else nan,
            "disc_acc_expert": float((~true_gen & correct).sum()) / n_exp if n_exp >= 1 else nan,
            "disc_acc_gen": float((true_gen & correct).sum()) / max(1.0, n_gen),
            "disc_entropy": float(ent),
            "disc_proportion_expert_true": n_exp / n_lab if n_lab > 0 else nan,
            "disc_proportion_expert_pred": n_exp_pred / n_lab if n_lab > 0 else nan,
            "n_expert": n_exp, "n_generated": n_gen,
        }


class _TorchCompatExpertIndices:
    """Index stream of the reference's expert loader: DataLoader(shuffle=True, drop_last=True) over
    the demonstrations, re-iterated forever by endless_iter (algorithms/base.py:272-282,
    util/util.py:215-241), INCLUDING the iterators endless_iter creates and drops, so the global
    torch RNG advances exactly as in the reference.  Only indices are produced (a range dataset);
    the rows are gathered on the device."""

    def __init__(self, n: int, batch_size: int):
        from torch.utils import data as th_data

        loader = th_data.DataLoader(range(n), batch_size=batch_size, shuffle=True, drop_last=True)
        probe = iter(loader)  # endless_iter: `iter(iterable) == iterable` check
        del probe
        next(iter(loader))    # get_first_iter_element
        self._it = itertools.chain.from_iterable(itertools.repeat(loader))

    def next(self) -> th.Tensor:
        return next(self._it).long()


class FusedAdamState:
    """Optimiser handle of the fused path (Adam moments are flat device vectors next to the
    parameters; the step itself happens inside `train_disc`)."""

    def __init__(self, n_params: int, device, lr=1e-3, betas=(0.9, 0.999), eps=1e-8, step_word: Optional[th.Tensor] = None):
        self.exp_avg = th.zeros(n_params, device=device)
        self.exp_avg_sq = th.zeros(n_params, device=device)
        self.hp = _lib.Adam(lr=lr, beta1=betas[0], beta2=betas[1], eps=eps)
        self.defaults = dict(lr=lr, betas=tuple(betas), eps=eps)
        # the step count (bias correction) lives in the device counter block so that captured graphs advance it;
        # `step_word` is the one-element int64 view of that word
        self.step_word = step_word

    def state_dict(self):
        step = int(self.step_word.item()) if self.step_word is not None else 0
        return {"exp_avg": self.exp_avg.clone(), "exp_avg_sq": self.exp_avg_sq.clone(), "defaults": dict(self.defaults),
                "step": step}

    def load_state_dict(self, sd):
        self.exp_avg.copy_(sd["exp_avg"])
        self.exp_avg_sq.copy_(sd["exp_avg_sq"])
        d = sd.get("defaults")
        if d:
            self.defaults = dict(lr=d["lr"], betas=tuple(d["betas"]), eps=d["eps"])
            self.hp = _lib.Adam(lr=d["lr"], beta1=d["betas"][0], beta2=d["betas"][1], eps=d["eps"])
        if self.step_word is not None and "step" in sd:  # warm moments with a cold bias correction would overshoot
            self.step_word.fill_(int(sd["step"]))

    def zero_grad(self):
        pass


class AdversarialTrainer(base.DemonstrationAlgorithm):
    """Base class for GAIL and AIRL."""

    def __init__(self, *, demonstrations, demo_batch_size: int, venv, gen_algo, reward_net,
                 demo_minibatch_size: Optional[int] = None, n_disc_updates_per_round: int = 2,
                 log_dir="output/", disc_opt_cls: Type[th.optim.Optimizer] = th.optim.Adam,
                 disc_opt_kwargs: Optional[Mapping] = None, gen_train_timesteps: Optional[int] = None,
                 gen_replay_buffer_capacity: Optional[int] = None, custom_logger=None,
                 init_tensorboard: bool = False, init_tensorboard_graph: bool = False,
                 debug_use_ground_truth: bool = False, allow_variable_horizon: bool = False,
                 sampling: str = "device", seed: int = 0):
        self.demo_batch_size = demo_batch_size
        self.demo_minibatch_size = demo_minibatch_size or demo_batch_size
        if self.demo_batch_size % self.demo_minibatch_size != 0:
            raise ValueError("Batch size must be a multiple of minibatch size.")
        if sampling not in ("device", "host_compat"):
            raise ValueError("sampling must be 'device' or 'host_compat'")
        self.sampling, self.seed = sampling, int(seed)
        self.venv = venv
        self.gen_algo = gen_algo
        self._device = th.device(gen_algo.device)
        self._reward_net: reward_nets.RewardNet = reward_net.to(self._device)
        self._expert_table = None
        self._expert_compat = None
        super().__init__(demonstrations=demonstrations, custom_logger=custom_logger,
                         allow_variable_horizon=allow_variable_horizon)
        self._global_step = 0
        self._disc_step = 0
        self.n_disc_updates_per_round = n_disc_updates_per_round
        self.debug_use_ground_truth = debug_use_ground_truth
        self._log_dir = log_dir
        if init_tensorboard or init_tensorboard_graph:
            self.logger.warn("TensorBoard summaries are not produced by the GPU trainer (logging is host I/O).")

        # -- discriminator network + optimiser -------------------------------------------------------------------
        self._fused_net = self._find_fused(self._reward_net)
        self._disc_opt_cls = disc_opt_cls
        self._disc_opt_kwargs = dict(disc_opt_kwargs or {})
        fusable_opt = (disc_opt_cls is th.optim.Adam and self._fused_net is not None
                       and set(self._disc_opt_kwargs) <= {"lr", "betas", "eps"})
        if fusable_opt:
            eng = self._fused_net.engine()
            self._disc_opt = FusedAdamState(eng.desc.n_params, self._device, **self._disc_opt_kwargs,
                                            step_word=self.venv.state[_lib.ST_DISC_STEP:_lib.ST_DISC_STEP + 1])
        else:
            self._disc_opt = disc_opt_cls(self._reward_net.parameters(), **self._disc_opt_kwargs)
        self._fused = fusable_opt

        # -- environment wrapping (common.py:227-241) ---------------------------------------------------------------
        self.venv_buffering = wrappers.BufferingWrapper(self.venv)
        if debug_use_ground_truth:
            self.venv_wrapped = self.venv_buffering
            self.gen_callback = None
        else:
            self.venv_wrapped = reward_wrapper.RewardVecEnvWrapper(self.venv_buffering,
                                                                   reward_fn=self.reward_train.predict_processed)
            self.gen_callback = self.venv_wrapped.make_log_callback()
        self.venv_train = self.venv_wrapped
        self.gen_algo.set_env(self.venv_train)
        self.gen_algo.set_logger(self.logger)

        if gen_train_timesteps is None:
            env = self.gen_algo.get_env()
            assert env is not None
            self.gen_train_timesteps = env.num_envs
            if hasattr(self.gen_algo, "n_steps"):
                self.gen_train_timesteps *= self.gen_algo.n_steps
        else:
            self.gen_train_timesteps = gen_train_timesteps
        if gen_replay_buffer_capacity is None:
            gen_replay_buffer_capacity = self.gen_train_timesteps
        self._gen_replay_buffer = buffer.ReplayBuffer(gen_replay_buffer_capacity, self.venv)
        self.venv_buffering.attach_ring(self._gen_replay_buffer)

        # -- static device buffers of one discriminator update ----------------------------------------------------
        B, mb = self.demo_batch_size, self.demo_minibatch_size
        v = self.venv
        self._tw = _desc.table_width(v.d_obs, v.d_act)
        self._bw = _desc.batch_rows(v.d_obs, v.d_act)
        self._ld = _desc.batch_ld(2 * mb)
        self._batch = th.zeros(self._bw, self._ld, device=self._device)
        self._logits = th.zeros(2 * mb, device=self._device)
        self._idx_e = th.zeros(B, dtype=th.int64, device=self._device)
        self._idx_g = th.zeros(B, dtype=th.int64, device=self._device)
        self._stats = th.zeros(16, device=self._device)
        self.disc_train_mode = False  # set by `train()`'s `networks.training(self.reward_train)`
        self._capturing = False
        self._graph = None
        self.use_cuda_graph = True   # replay warm kernel sequences from CUDA graphs (device sampling only)
        # GAIL: a discriminator update needs the round's rollouts but not the PPO update (which needs the rollouts but
        # not the discriminator), so the two run concurrently: the PPO kernel occupies the 8 SMs of one cluster, the
        # discriminator kernels the rest.  Results are bit-identical to the serial order.  AIRL's logit needs
        # log pi of the UPDATED policy (common.py:606-615), so it stays on one stream.
        self.overlap_disc_with_gen = True
        self._disc_stream = None
        self._ev_disc = None
        self._disc_graphs = {}
        self._stage = {}
        # SURVEY App. A.14: the reference evaluates `policy.evaluate_actions` on every discriminator minibatch (GAIL
        # discards the result, common.py:606-615) with the policy still in the train mode SB3's PPO.train left it in,
        # so a NormalizeFeaturesExtractor's RunningNorm also sees the expert|generator observations.  Reproduced: the
        # batch moments are computed beside the discriminator update and folded into the policy's statistics, in
        # order, once the PPO update (which updates the same statistics) has finished.
        self.reproduce_evaluate_actions_side_effect = True
        self._pn_cap = 256
        self._pn_defer = None    # [4 + cap * (2 d_obs + 1)] slot list of deferred batch moments
        self._pn_pending = 0     # host mirror of the number of slots in use
        self._ev_fold = None
        # multi-GPU (set_distributed): the discriminator is the GLOBAL-batch discriminator -- every optimiser step
        # all-reduces [gradients | statistic sums] and all-gathers the RunningNorm batch moments, so the replicas apply
        # bit-identical updates (SURVEY 8e; reference loss = mean over the global 2 * minibatch rows, common.py:360-368)
        self._dist_group = None
        self._dist_world = 1
        self._stats_pub = None   # pinned host mirror of the nine statistics + sequence word (imb_stats_publish)
        self._stats_pub_i = None
        self._pub_seq = None
        self._dn_local = None    # my batch moments (one slot)
        self._dn_all = None      # the gathered slot list

    # -- helpers --------------------------------------------------------------------------------------------------
    @staticmethod
    def _find_fused(net):
        while net is not None and not hasattr(net, "_engine"):
            net = getattr(net, "base", None) if isinstance(net, reward_nets.RewardNetWrapper) else None
        return net

    @property
    def policy(self):
        policy = self.gen_algo.policy
        assert policy is not None
        return policy

    @abc.abstractmethod
    def logits_expert_is_high(self, state, action, next_state, done, log_policy_act_prob=None) -> th.Tensor:
        """Discriminator logits; high = expert-like."""

    @property
    @abc.abstractmethod
    def reward_train(self) -> reward_nets.RewardNet:
        """Reward used to train generator policy."""

    @property
    @abc.abstractmethod
    def reward_test(self) -> reward_nets.RewardNet:
        """Reward used at test time."""

    _needs_logp = False  # AIRL sets True

    # -- demonstrations (common.py:306-315; algorithms/base.py:226-288) --------------------------------------------------
    def set_demonstrations(self, demonstrations) -> None:
        tr = types.as_transition_arrays(demonstrations)
        n = len(tr["obs"])
        if self.demo_batch_size <= 0:
            raise ValueError(f"batch_size={self.demo_batch_size} must be positive.")
        if n < self.demo_batch_size:
            raise ValueError(f"Number of transitions in `demonstrations` {n} is smaller than batch size "
                             f"{self.demo_batch_size}.")
        self._expert_table = self._rows_to_table(tr)
        self._expert_n = n
        self._expert_state = th.zeros(_lib.ST_WORDS, dtype=th.int64, device=self._device)
        self._expert_compat = (_TorchCompatExpertIndices(n, self.demo_batch_size)
                               if self.sampling == "host_compat" else None)
        # captured graphs hold the OLD table / sampling-state pointers: drop them (they are re-captured on demand)
        if getattr(self, "_disc_graphs", None):
            self._disc_graphs = {}
        if getattr(self, "_graph", None) is not None:
            self._graph = None

    def _rows_to_table(self, tr: Mapping[str, np.ndarray]) -> th.Tensor:
        """host/device transition arrays -> AoS device table (RewardNet.preprocess semantics)."""
        v, dev = self.venv, self._device
        n = len(tr["obs"])

        def f32(x):
            return th.as_tensor(np.ascontiguousarray(x) if isinstance(x, np.ndarray) else x).to(dev).float().reshape(n, -1).contiguous()
        table = th.zeros(n, _desc.table_width(v.d_obs, v.d_act), device=dev)
        st = th.zeros(_lib.ST_WORDS, dtype=th.int64, device=dev)
        dones = th.as_tensor(np.asarray(tr["dones"]) if not isinstance(tr["dones"], th.Tensor) else tr["dones"])
        dones = dones.to(dev).to(th.uint8).contiguous()
        if v.discrete:
            acts = th.as_tensor(np.asarray(tr["acts"]) if not isinstance(tr["acts"], th.Tensor) else tr["acts"])
            _lib.table_store(table, n, v.d_obs, v.d_act, f32(tr["obs"]), None, acts.to(dev).long().reshape(n).contiguous(),
                             f32(tr["next_obs"]), dones, n, False, st)
        else:
            _lib.table_store(table, n, v.d_obs, v.d_act, f32(tr["obs"]), f32(tr["acts"]), None, f32(tr["next_obs"]),
                             dones, n, False, st)
        return table

    # -- generator update and discriminator updates on two streams (GAIL) -------------------------------------------
    def _overlap(self) -> bool:
        return bool(self._fused and self.overlap_disc_with_gen and not self._needs_logp and self._device.type == "cuda")

    def _disc_ctx(self):
        """Stream context of the discriminator updates: a side stream that starts from the generator's "rollout done"
        event (no-op context when the overlap is off, e.g. AIRL)."""
        if not self._overlap():
            return contextlib.nullcontext()
        if self._disc_stream is None:
            self._disc_stream = th.cuda.Stream(device=self._device)
            self._ev_disc = th.cuda.Event()
        self._disc_stream.wait_event(self.gen_algo.ev_rollout)
        return th.cuda.stream(self._disc_stream)

    def join(self) -> None:
        """Order the current stream after every discriminator update enqueued so far (callers of `train_disc_async`
        that go on to touch the reward network on the current stream, e.g. the multi-GPU round sync)."""
        self._join_disc()
        self._fold_policy_norm()

    def _join_disc(self) -> None:
        """Make the current stream wait for the discriminator updates enqueued so far (the next rollout relabels its
        rewards with the updated reward network)."""
        if self._disc_stream is not None and self._ev_disc is not None:
            th.cuda.current_stream().wait_event(self._ev_disc)

    # -- discriminator update -------------------------------------------------------------------------------------------
    def _sample_expert_indices(self) -> None:
        if self._expert_compat is not None:
            self._idx_e.copy_(self._expert_compat.next())
        else:
            _lib.sample_indices(1, self._idx_e, self.demo_batch_size, self._expert_n, self.seed, self._expert_state)

    def _sample_gen_indices(self) -> None:
        if self.sampling == "host_compat":
            size = self._gen_replay_buffer.size()
            self._idx_g.copy_(th.as_tensor(np.random.randint(size, size=self.demo_batch_size)))
        else:
            _lib.sample_indices(0, self._idx_g, self.demo_batch_size, 0, self.seed, self.venv.state)

    # -- host-provided samples: async copies into persistent staging buffers ------------------------------------
    def _stage_host(self, samples: Mapping, which: str) -> None:
        """H2D (non-blocking when the source is pinned) of obs/acts/next_obs/dones into static device
        buffers; the AoS packing (imb_table_store) is part of the update's kernel sequence."""
        v, dev, B = self.venv, self._device, self.demo_batch_size
        st = self._stage.get(which)
        if st is None:
            st = dict(obs=th.empty(B, v.d_obs, device=dev), next_obs=th.empty(B, v.d_obs, device=dev),
                      acts=(th.empty(B, dtype=th.int64, device=dev) if v.discrete else th.empty(B, v.d_act, device=dev)),
                      dones=th.empty(B, dtype=th.uint8, device=dev),
                      table=th.zeros(B, _desc.table_width(v.d_obs, v.d_act), device=dev),
                      state=th.zeros(_lib.ST_WORDS, dtype=th.int64, device=dev))
            self._stage[which] = st
        for k in ("obs", "next_obs", "acts", "dones"):
            src = samples[k]
            dst = st[k]
            if type(src) is th.Tensor and src.dtype == dst.dtype and src.shape == dst.shape and not src.requires_grad:
                dst.copy_(src, non_blocking=True)  # (the common case of the hot loop: a ready host / device tensor)
                continue
            if isinstance(src, np.ndarray):
                src = th.from_numpy(np.ascontiguousarray(src) if src.flags.writeable else src.copy())
            dst = st[k]
            src = src.detach().reshape(dst.shape)
            if src.dtype != dst.dtype and not src.is_cuda:
                src = src.to(dst.dtype)  # host-side cast (bool -> uint8, float64 -> float32, ...)
            dst.copy_(src, non_blocking=True)

    def _pack_staged(self, which: str) -> th.Tensor:
        v, st, B = self.venv, self._stage[which], self.demo_batch_size
        _lib.table_store(st["table"], B, v.d_obs, v.d_act, st["obs"], None if v.discrete else st["acts"],
                         st["acts"] if v.discrete else None, st["next_obs"], st["dones"], B, False, st["state"])
        return st["table"]

    def train_disc_async(self, *, expert_samples: Optional[Mapping] = None, gen_samples: Optional[Mapping] = None,
                         stats_out: Optional[th.Tensor] = None, check_ring: bool = True) -> th.Tensor:
        """One discriminator update entirely on the stream; returns the device stats vector
        (index order = STAT_KEYS) without synchronising.  The kernel sequence after the H2D copies is
        replayed from a CUDA graph once warm (device sampling only)."""
        if not self._fused:
            raise NotImplementedError("train_disc_async needs the fused Adam path")
        if gen_samples is None and check_ring and self._gen_replay_buffer.size() == 0:
            raise RuntimeError("No generator samples for training. Call `train_gen()` first.")
        if self._capturing:  # (whole-round capture: the caller forks / joins the streams itself)
            return self._train_disc_async_on_stream(expert_samples, gen_samples, stats_out)
        with self._disc_ctx():
            out = self._train_disc_async_on_stream(expert_samples, gen_samples, stats_out)
            if self._disc_stream is not None and self._overlap():
                self._ev_disc.record(self._disc_stream)
        return out

    def _train_disc_async_on_stream(self, expert_samples, gen_samples, stats_out) -> th.Tensor:
        e_host, g_host = expert_samples is not None, gen_samples is not None
        if (not self._capturing and self._pn_pending + self.demo_batch_size // self.demo_minibatch_size > self._pn_cap):
            self.join()  # (hundreds of updates without a train_gen in between: make room in the slot list)
        if e_host:
            self._stage_host(self._check_samples(expert_samples, "expert"), "expert")
        if g_host:
            self._stage_host(self._check_samples(gen_samples, "gen"), "gen")
        train_mode = bool(self.reward_train.training or self.disc_train_mode)
        out = self._stats if stats_out is None else stats_out
        graphable = (self.use_cuda_graph and not self._capturing and self.sampling == "device"
                     and (e_host or self._expert_compat is None))
        if not graphable:
            self._disc_update_body(e_host, g_host, train_mode, out)
        else:
            eng = self._fused_net.engine()
            key = (e_host, g_host, train_mode, out.data_ptr(), eng.params.data_ptr(), eng.norm_state.data_ptr(),
                   self._gen_replay_buffer.table.data_ptr(),
                   self.policy.flat_vectors()[0].data_ptr() if self._needs_logp else 0)
            ent = self._disc_graphs.get(key)
            if ent is None:
                # first call with this signature runs eagerly (allocations, function attributes) ...
                self._disc_update_body(e_host, g_host, train_mode, out)
                self._disc_graphs[key] = "warm"
            else:
                if ent == "warm":  # ... the second one is captured, later ones are replayed
                    before = _lib.LAUNCHES["count"]
                    self._capturing = True
                    try:
                        g = th.cuda.CUDAGraph()
                        with th.cuda.graph(g):
                            self._disc_update_body(e_host, g_host, train_mode, out)
                    finally:
                        self._capturing = False
                    ent = (g, _lib.LAUNCHES["count"] - before)
                    _lib.LAUNCHES["count"] = before
                    self._disc_graphs[key] = ent
                ent[0].replay()
                _lib.LAUNCHES["count"] += ent[1]
        if not self._capturing:
            self._disc_step += 1
            if self._side_effect_active() and self._overlap():
                self._pn_pending += self.demo_batch_size // self.demo_minibatch_size
            if out is self._stats and self._pub_seq is not None:
                self._pub_seq += 1  # (one Adam step per update; wraps like the int32 mirror does -- never in practice)
        return out

    def _disc_update_body(self, e_host: bool, g_host: bool, train_mode: bool, out: th.Tensor) -> None:
        B, mb = self.demo_batch_size, self.demo_minibatch_size
        eng = self._fused_net.engine()
        opt: FusedAdamState = self._disc_opt
        # device sampling on both sides: index generation and both gathers are ONE launch per minibatch
        fused_sampling = (not e_host and not g_host and self.sampling == "device" and self._expert_compat is None)
        if fused_sampling:
            ring = self._gen_replay_buffer
        elif not e_host:
            self._sample_expert_indices()
            e_table, e_idx, e_cap = self._expert_table, self._idx_e, self._expert_n
        else:
            e_table, e_idx, e_cap = self._pack_staged("expert"), None, B
        if fused_sampling:
            pass
        elif not g_host:
            self._sample_gen_indices()
            g_table, g_idx, g_cap = self._gen_replay_buffer.table, self._idx_g, self._gen_replay_buffer.capacity
        else:
            g_table, g_idx, g_cap = self._pack_staged("gen"), None, B
        n = 2 * mb
        starts = list(range(0, B, mb))
        for i, start in enumerate(starts):
            if fused_sampling:
                _lib.disc_sample_gather(self._expert_table, self._expert_n, ring.table, ring.capacity, self._tw, mb, start,
                                        self.seed, self._expert_state, self.venv.state, self._batch, self._ld)
            else:
                ei = e_idx[start:start + mb] if e_idx is not None else None
                gi = g_idx[start:start + mb] if g_idx is not None else None
                et = e_table if e_idx is not None else e_table[start:start + mb]
                gt = g_table if g_idx is not None else g_table[start:start + mb]
                _lib.gather_rows(et, e_cap if e_idx is not None else mb, self._tw, ei, mb, self._batch, self._ld, 0)
                _lib.gather_rows(gt, g_cap if g_idx is not None else mb, self._tw, gi, mb, self._batch, self._ld, mb)
            self._policy_norm_side_effect(eng, n)
            if self._needs_logp:
                pp, pn, _ = self.policy.flat_vectors()
                _lib.policy_logp(self.policy.desc, pp, pn, self._batch, self._ld, n, self._bw - 1)
            tn = train_mode and eng.has_norm
            W = self._dist_world
            if tn and W > 1:
                self._global_norm_update(eng, n)
            elif tn:
                eng.norm_update(self._batch, self._ld, n)
            eng.fwd_bwd(self._batch, self._ld, n, mb, 1.0 / (2 * B * W), None, self._logits, i == 0, tn)
            if i + 1 < len(starts):
                eng.reduce(None)
            elif W > 1:  # global-batch step: sum [gradients | statistic sums] over the ranks, identical Adam everywhere
                import torch.distributed as dist

                eng.reduce(None)
                k = (eng.desc.n_params + 31) // 32 * 32 + 5
                dist.all_reduce(eng.ws[:k], op=dist.ReduceOp.SUM, group=self._dist_group)
                _lib.disc_set_rows(eng.desc, eng.ws, n * W, mb * W)
                _lib.disc_adam(eng.desc, opt.hp, eng.params, opt.exp_avg, opt.exp_avg_sq, None, 1.0, eng.ws,
                               self.venv.state, out)
            else:  # last minibatch: reduction, optimiser step and the statistics in one launch
                _lib.disc_reduce_adam(eng.desc, opt.hp, eng.params, opt.exp_avg, opt.exp_avg_sq, 1.0, eng.ws,
                                      self.venv.state, out)
        if fused_sampling:
            _lib.sample_advance2(B, self._expert_n, self._expert_state, self.venv.state)
        if out is self._stats:  # the synchronous API reads these nine floats: publish them to host-mapped memory
            if self._stats_pub is None:
                self._stats_pub = th.zeros(16, dtype=th.float32).pin_memory()
                self._stats_pub_i = self._stats_pub.numpy().view(np.int32)
                self._stats_pub_i[15] = -1
                self._pub_seq = None
            _lib.stats_publish(out, 9, self._stats_pub, self.venv.state, _lib.ST_DISC_STEP)

    def _global_norm_update(self, eng, n: int) -> None:
        """RunningNorm.update_stats with the GLOBAL minibatch: local moments -> all-gather -> the W batches are folded in
        rank order on every rank (identical arithmetic, identical result)."""
        import torch.distributed as dist

        d = eng.desc
        slot = 2 * d.base.din + 1
        _lib.norm_batch_stats(d, self._batch, self._ld, n, 0, d.base.din, eng.norm_state, eng.norm_count,
                              self._dn_local, 1, eng.ws)
        dist.all_gather_into_tensor(self._dn_all[4:], self._dn_local[4:4 + slot], group=self._dist_group)
        _lib.norm_fold(d.base.din, self._dn_all, eng.norm_state, eng.norm_count, self._dist_world)

    # -- multi-GPU -----------------------------------------------------------------------------------------------------------
    def set_distributed(self, group=None) -> None:
        """One process per GPU (`torch.distributed` initialised): shard = this trainer's env slice, ring and sampling
        streams; discriminator steps become global-batch steps (see __init__).  The generator side is synchronised by
        `imitation_b200.distributed.trainer_round_sync(self)` once per round."""
        import torch.distributed as dist

        if not self._fused:
            raise NotImplementedError("distributed training needs the fused Adam path")
        d = self._fused_net.engine().desc
        if d.shaped or d.use_next_state or d.use_done:
            raise NotImplementedError("distributed discriminator steps: BasicRewardNet(state, action) only")
        self._dist_group = group
        self._dist_world = dist.get_world_size(group)
        slot = 2 * d.base.din + 1
        self._dn_local = th.zeros(4 + slot, device=self._device)
        self._dn_all = th.zeros(4 + self._dist_world * slot, device=self._device)
        self._disc_graphs = {}
        self._graph = None
        # the replicas start from rank 0's discriminator (parameters, Adam state, RunningNorm statistics, step counter)
        eng, opt = self._fused_net.engine(), self._disc_opt
        for t in (eng.params, opt.exp_avg, opt.exp_avg_sq, eng.norm_state, eng.norm_count,
                  self.venv.state[_lib.ST_DISC_STEP:_lib.ST_DISC_STEP + 1]):
            dist.broadcast(t, 0, group=group)

    # -- SURVEY App. A.14 --------------------------------------------------------------------------------------------------
    def _side_effect_active(self) -> bool:
        pol = self.gen_algo.policy
        return bool(self.reproduce_evaluate_actions_side_effect and getattr(pol, "normalize_features", False)
                    and self._fused and getattr(pol, "training", True))

    def _policy_norm_side_effect(self, eng, n: int) -> None:
        """RunningNorm.update_stats of the policy's feature extractor on the observations of the current discriminator
        minibatch (batch rows [0, d_obs)).  Serial path (AIRL): immediately, before log pi is evaluated -- exactly where
        `evaluate_actions` does it.  Two-stream path (GAIL): moments now, fold after the PPO update (`_fold_policy_norm`)."""
        if not self._side_effect_active():
            return
        pol = self.gen_algo.policy
        _, pn, pc = pol.flat_vectors()
        if not self._overlap():
            _lib.norm_batch_stats(eng.desc, self._batch, self._ld, n, 0, pol.d_obs, pn, pc, None, 0, eng.ws)
            return
        if self._pn_defer is None:
            self._pn_defer = th.zeros(4 + self._pn_cap * (2 * pol.d_obs + 1), device=self._device)
        _lib.norm_batch_stats(eng.desc, self._batch, self._ld, n, 0, pol.d_obs, pn, pc, self._pn_defer, self._pn_cap,
                              eng.ws)

    def _fold_policy_norm(self) -> None:
        """Apply the deferred moments on the CURRENT stream (ordered after the PPO update by stream order and after the
        discriminator stream by `_join_disc`)."""
        if self._pn_defer is None or (self._pn_pending == 0 and not self._capturing):
            return
        pol = self.gen_algo.policy
        _, pn, pc = pol.flat_vectors()
        _lib.norm_fold(pol.d_obs, self._pn_defer, pn, pc)
        self._pn_pending = 0
        if not self._capturing and self._disc_stream is not None:  # later updates append to the emptied slot list
            if self._ev_fold is None:
                self._ev_fold = th.cuda.Event()
            self._ev_fold.record()
            self._disc_stream.wait_event(self._ev_fold)

    # -- whole round as one CUDA graph (no host work between kernels) ---------------------------------------------
    def _enqueue_round(self) -> None:
        gen = self.gen_algo
        gen.collect_rollouts()
        side = None
        if self._overlap():  # fork: the discriminator updates run beside the PPO update (two branches of the graph)
            if self._disc_stream is None:
                self._disc_stream = th.cuda.Stream(device=self._device)
                self._ev_disc = th.cuda.Event()
            side = self._disc_stream
            fork = th.cuda.Event()
            fork.record()
            side.wait_event(fork)
        gen.train()
        self.disc_train_mode = True
        try:
            with (th.cuda.stream(side) if side is not None else contextlib.nullcontext()):
                for k in range(self.n_disc_updates_per_round):
                    self.train_disc_async(stats_out=self._round_stats[k], check_ring=False)
        finally:
            self.disc_train_mode = False
        if side is not None:  # join
            done = th.cuda.Event()
            done.record(side)
            th.cuda.current_stream().wait_event(done)
            if self._side_effect_active() and self._pn_defer is not None:
                self._fold_policy_norm()

    def capture_round(self) -> None:
        """Capture [rollout -> GAE -> PPO update -> n_disc x discriminator update] into a CUDA graph.
        Needs device-side sampling (all counters live in the device state block) and at least one
        eager round before (buffers allocated, function attributes set)."""
        if not (self._fused and self.sampling == "device"):
            raise NotImplementedError("graph capture needs the fused Adam path and sampling='device'")
        if self.gen_algo._tbl is None:
            raise RuntimeError("run one eager round (train_gen + train_disc) before capture_round()")
        self._round_stats = th.zeros(self.n_disc_updates_per_round, 16, device=self._device)
        before = _lib.LAUNCHES["count"]
        self._capturing = self.gen_algo._capturing = True
        try:
            g = th.cuda.CUDAGraph()
            with th.cuda.graph(g):
                self._enqueue_round()
        finally:
            self._capturing = self.gen_algo._capturing = False
        self._graph = g
        self._graph_launches = _lib.LAUNCHES["count"] - before
        _lib.LAUNCHES["count"] = before

    def replay_round(self) -> th.Tensor:
        """Run one captured round; returns the device stats [n_disc][16] (no synchronisation)."""
        t0 = self.venv.host_ep_step
        self._join_disc()
        self._graph.replay()
        _lib.LAUNCHES["count"] += self._graph_launches
        self.gen_algo.after_rollout_host(t0)
        self.venv_buffering.discard()
        self._global_step += 1
        self._disc_step += self.n_disc_updates_per_round
        self._pub_seq = None  # (the replayed updates advanced the device's step count without publishing)
        return self._round_stats

    def _check_samples(self, samples: Mapping, who: str) -> Mapping:
        d = dict(samples)
        for k in ("obs", "acts", "next_obs", "dones"):
            if isinstance(d[k], th.Tensor):
                d[k] = d[k].detach()
        return d

    def train_disc(self, *, expert_samples: Optional[Mapping] = None, gen_samples: Optional[Mapping] = None
                   ) -> Mapping[str, float]:
        """Perform a single discriminator update (common.py:317-389)."""
        B = self.demo_batch_size
        n_e = len(expert_samples["obs"]) if expert_samples is not None else B
        if gen_samples is None and self._gen_replay_buffer.size() == 0:
            raise RuntimeError("No generator samples for training. Call `train_gen()` first.")
        n_g = len(gen_samples["obs"]) if gen_samples is not None else B
        if not (n_g == n_e == B):
            raise ValueError("Need to have exactly `demo_batch_size` number of expert and generator samples, each. "
                             f"(n_gen={n_g} n_expert={n_e} demo_batch_size={B})")
        with self.logger.accumulate_means("disc"):
            if self._fused:
                stats_t = self.train_disc_async(expert_samples=expert_samples, gen_samples=gen_samples,
                                                check_ring=False)
                vals = self._read_stats(stats_t)  # the one D2H read the Mapping[str, float] return needs
                train_stats = {k: float(v) for k, v in zip(STAT_KEYS, vals)}
            else:
                train_stats = self._train_disc_generic(expert_samples, gen_samples)
            self.logger.record("global_step", self._global_step)
            for k, v in train_stats.items():
                self.logger.record(k, v)
            self.logger.dump(self._disc_step)
        return train_stats

    def _read_stats(self, stats_t: th.Tensor) -> np.ndarray:
        """Nine floats device -> pinned host on the stream that produced them (does not wait for the PPO update on the
        other stream); waits on an event instead of a device-wide synchronisation."""
        if stats_t is self._stats and self._stats_pub is not None:
            # the update's last kernel wrote the statistics and then the Adam step count into host-mapped memory: poll
            # the word until it shows the step this update produces (`_pub_seq` = step expected after every update
            # issued so far, advanced on the host by `_train_disc_async_on_stream`)
            seq = self._stats_pub_i
            if self._pub_seq is not None:
                import time as _time

                t0 = None
                while int(seq[15]) != self._pub_seq:
                    if t0 is None:
                        t0 = _time.perf_counter()
                    elif _time.perf_counter() - t0 > 0.5:
                        break  # (e.g. the step counter was restored from a checkpoint: resynchronise below)
                else:
                    return self._stats_pub.numpy()[:9].copy()
            # first read or resynchronisation: wait for the stream, then learn the device's step count from the mirror
            (self._disc_stream if (self._disc_stream is not None and self._overlap()) else th.cuda.current_stream()).synchronize()
            self._pub_seq = int(seq[15])
            return self._stats_pub.numpy()[:9].copy()
        if getattr(self, "_stats_host", None) is None:
            self._stats_host = th.empty(9, dtype=th.float32).pin_memory()
            self._ev_stats = th.cuda.Event()
        with self._disc_ctx():
            self._stats_host.copy_(stats_t[:9], non_blocking=True)
            self._ev_stats.record()
        self._ev_stats.synchronize()
        return self._stats_host.numpy().copy()

    def _train_disc_generic(self, expert_samples, gen_samples) -> Mapping[str, float]:
        """Any torch optimiser: logits through the fused autograd Function, BCE/optimiser in torch."""
        B, mb = self.demo_batch_size, self.demo_minibatch_size
        v = self.venv

        def rows(samples, idx_fn, table, cap):
            if samples is not None:
                return self._rows_to_table(self._check_samples(samples, ""))
            idx_fn()
            return None
        e_rows = rows(expert_samples, self._sample_expert_indices, None, None)
        if e_rows is None:
            e_rows = self._expert_table[self._idx_e]
        g_rows = rows(gen_samples, self._sample_gen_indices, None, None)
        if g_rows is None:
            g_rows = self._gen_replay_buffer.table[self._idx_g]
        self._disc_opt.zero_grad()
        Do, Da = v.d_obs, v.d_act
        for start in range(0, B, mb):
            r = th.cat([e_rows[start:start + mb], g_rows[start:start + mb]])
            state, action = r[:, :Do], r[:, Do:Do + Da]
            next_state, done = r[:, Do + Da:2 * Do + Da], r[:, -1]
            labels = th.cat([th.ones(mb, device=r.device), th.zeros(mb, device=r.device)])
            logp = None
            if self._needs_logp:
                with th.no_grad():
                    acts = action.argmax(1) if v.discrete else action
                    logp = self.policy.evaluate_actions(state, acts)[1].reshape(2 * mb)
            logits = self.logits_expert_is_high(state, action, next_state, done, logp)
            loss = F.binary_cross_entropy_with_logits(logits, labels) * (mb / B)
            loss.backward()
        self._disc_opt.step()
        self._disc_step += 1
        return compute_train_stats(logits.detach(), labels.long(), loss.detach())

    # -- generator -------------------------------------------------------------------------------------------------------
    def train_gen(self, total_timesteps: Optional[int] = None, learn_kwargs: Optional[Mapping] = None) -> None:
        """gen_algo.learn + pop/flatten/store (common.py:391-425); the store is fused into the rollout."""
        if total_timesteps is None:
            total_timesteps = self.gen_train_timesteps
        self._join_disc()  # the rollouts are relabelled with the reward network the previous updates produced
        self._fold_policy_norm()
        with self.logger.accumulate_means("gen"):
            self.gen_algo.learn(total_timesteps=total_timesteps, reset_num_timesteps=False,
                                callback=self.gen_callback, **(learn_kwargs or {}))
            self._global_step += 1
        ep_lens = list(self.venv_buffering._ep_lens)
        self.venv_buffering.discard()  # the samples were consumed by the fused ring store
        self._check_fixed_horizon(ep_lens)

    def train(self, total_timesteps: int, callback: Optional[Callable[[int], None]] = None) -> None:
        """Alternate generator and discriminator training (common.py:427-461)."""
        n_rounds = total_timesteps // self.gen_train_timesteps
        assert n_rounds >= 1, ("No updates (need at least "
                               f"{self.gen_train_timesteps} timesteps, have only total_timesteps={total_timesteps})!")
        for r in range(n_rounds):
            self.train_gen(self.gen_train_timesteps)
            for _ in range(self.n_disc_updates_per_round):
                with networks.training(self.reward_train):
                    self.train_disc()
            if self._pn_pending:
                self.join()
            if callback:
                callback(r)
            self.logger.dump(self._global_step)
