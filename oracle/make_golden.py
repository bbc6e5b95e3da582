"""Generate tests/golden/*.npz by running the REFERENCE's own modules on seeded inputs.

TEST INFRASTRUCTURE.  Runs only in the build container (needs /root/reference):
    python -m oracle.make_golden
The reference is imported unchanged from /root/reference/src through the names-only
shim (oracle/_shim); every stored output is produced by reference code:
  algorithms/adversarial/{common,gail,airl}.py, rewards/reward_nets.py, util/networks.py,
  data/{buffer,wrappers,rollout,serialize,types}.py, rewards/{reward_wrapper,serialize}.py, algorithms/base.py,
  algorithms/preference_comparisons.py, util/util.py.
The fixtures pin (a) the CPU restatement in oracle/*_port.py and (b) the CUDA path.
"""
import os
import sys

import numpy as np
import torch as th

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
from oracle import refimport, synth_env  # noqa: E402
from oracle.api_cases import (HORIZON_SCRIPTS, PREF_SETTINGS, ROLLOUT_LENS, SAMPLE_UNTIL, SAMPLE_UNTIL_BAD,  # noqa: E402
                              SCHEDULE_RUNS, error, make_dataset_trajectories, make_hf_trajectories,
                              make_rollout_trajectories, validation_cases)

refimport.load()
from gymnasium import spaces  # noqa: E402  (shim)
from imitation.algorithms.adversarial import airl as ref_airl  # noqa: E402
from imitation.algorithms.adversarial import common as ref_common  # noqa: E402
from imitation.algorithms.adversarial import gail as ref_gail  # noqa: E402
from imitation.algorithms import base as ref_base  # noqa: E402
from imitation.data import buffer as ref_buffer  # noqa: E402
from imitation.data import rollout as ref_rollout  # noqa: E402
from imitation.data import types as ref_types  # noqa: E402
from imitation.data import wrappers as ref_wrappers  # noqa: E402
from imitation.rewards import reward_nets as ref_nets  # noqa: E402
from imitation.rewards import reward_wrapper as ref_rw  # noqa: E402
from imitation.util import logger as ref_logger  # noqa: E402
from imitation.util import networks as ref_networks  # noqa: E402
from imitation.util import util as ref_util  # noqa: E402
from stable_baselines3.common import policies as sb_policies  # noqa: E402
from stable_baselines3.common.on_policy_algorithm import OnPolicyAlgorithm  # noqa: E402
from stable_baselines3.common.vec_env import VecEnv  # noqa: E402

OUT = os.path.join(os.path.dirname(HERE), "tests", "golden")


class _FixedLogpPolicy(sb_policies.ActorCriticPolicy):
    """Stochastic-policy stand-in: log pi(a|s) = -0.5|a - M s|^2 - 1 (deterministic fn)."""

    def __init__(self, d_obs, d_act, seed=0):
        super().__init__()
        g = th.Generator().manual_seed(seed)
        self.M = th.randn(d_act, d_obs, generator=g) * 0.3

    def evaluate_actions(self, obs, acts):
        obs = obs.float()
        acts = acts.float()
        if acts.ndim == 1:
            acts = acts[:, None]
        mean = obs @ self.M.T[:, : acts.shape[1]]
        logp = -0.5 * ((acts - mean) ** 2).sum(1) - 1.0
        return None, logp, None


class _DummyGen(OnPolicyAlgorithm):
    def __init__(self, venv, policy, n_steps=4):
        self.env = venv
        self.policy = policy
        self.n_steps = n_steps
        self.device = th.device("cpu")


class _HostVenv(VecEnv):
    """Adapter: oracle SynthVecEnv under the (shim) SB3 VecEnv base class."""

    def __init__(self, inner):
        super().__init__(inner.num_envs, inner.observation_space, inner.action_space)
        self.inner = inner

    def reset(self):
        return self.inner.reset()

    def step_async(self, a):
        self.inner.step_async(a)

    def step_wait(self):
        return self.inner.step_wait()


def _state(module):
    return {k: v.detach().cpu().numpy().copy() for k, v in module.state_dict().items()}


def _flat(prefix, d):
    return {f"{prefix}/{k}": v for k, v in d.items()}


def _rand_transitions(rng, n, d_obs, d_act, discrete=False):
    obs = rng.standard_normal((n, d_obs)).astype(np.float32) * 1.5 + 0.3
    nobs = rng.standard_normal((n, d_obs)).astype(np.float32)
    acts = rng.integers(0, d_act, n) if discrete else rng.uniform(-1, 1, (n, d_act)).astype(np.float32)
    dones = rng.random(n) < 0.1
    return dict(obs=obs, acts=acts, next_obs=nobs, dones=dones)


def disc_case(name, algo, d_obs, d_act, discrete, net_kwargs, B, mb, steps, seed, shaped=False):
    th.manual_seed(seed)
    rng = np.random.default_rng(seed)
    obs_space = spaces.Box(-np.inf, np.inf, (d_obs,), np.float32)
    act_space = spaces.Discrete(d_act) if discrete else spaces.Box(-1, 1, (d_act,), np.float32)
    spec = synth_env.SynthEnvSpec(d_obs, d_act, discrete=discrete, horizon=50, seed=seed)
    venv = _HostVenv(synth_env.SynthVecEnv(spec, 4, spaces_mod=spaces))
    cls = ref_nets.BasicShapedRewardNet if shaped else ref_nets.BasicRewardNet
    net = cls(obs_space, act_space, **net_kwargs)
    policy = _FixedLogpPolicy(d_obs, 1 if discrete else d_act, seed)
    demos = _rand_transitions(rng, 4 * B, d_obs, d_act, discrete)
    demos_t = ref_types.Transitions(infos=np.array([{}] * (4 * B)), **demos)
    trainer_cls = ref_airl.AIRL if algo == "airl" else ref_gail.GAIL
    trainer = trainer_cls(demonstrations=demos_t, demo_batch_size=B, demo_minibatch_size=mb, venv=venv,
                          gen_algo=_DummyGen(venv, policy), reward_net=net,
                          custom_logger=ref_logger.configure(folder="/tmp/imb_golden_log", format_strs=[]))
    out = dict(meta=np.array([d_obs, d_act, int(discrete), B, mb, steps, seed]))
    out.update(_flat("init", _state(net)))
    for s in range(steps):
        ex = _rand_transitions(rng, B, d_obs, d_act, discrete)
        ge = _rand_transitions(rng, B, d_obs, d_act, discrete)
        ge["obs"] = ge["obs"] * 0.5 - 0.2
        with ref_networks.training(trainer.reward_train):
            stats = trainer.train_disc(expert_samples=ex, gen_samples=ge)
        out.update(_flat(f"step{s}/expert", ex))
        out.update(_flat(f"step{s}/gen", ge))
        out[f"step{s}/stats"] = np.array([stats[k] for k in sorted(stats)], np.float64)
        out.update(_flat(f"step{s}/state", _state(net)))
        # logits of the last minibatch, recomputed in eval mode with post-step params
        q = _rand_transitions(rng, 32, d_obs, d_act, discrete)
        out.update(_flat(f"step{s}/query", q))
        out[f"step{s}/reward_train"] = trainer.reward_train.predict_processed(
            q["obs"], q["acts"], q["next_obs"], q["dones"], update_stats=False) if algo == "airl" else \
            trainer.reward_train.predict_processed(q["obs"], q["acts"], q["next_obs"], q["dones"])
        out[f"step{s}/reward_test"] = trainer.reward_test.predict(q["obs"], q["acts"], q["next_obs"], q["dones"])
        s_th, a_th, ns_th, d_th = net.preprocess(q["obs"], q["acts"], q["next_obs"], q["dones"])
        with th.no_grad(), ref_networks.evaluating(net):
            logp = policy.evaluate_actions(th.as_tensor(q["obs"]), th.as_tensor(q["acts"]))[1]
            out[f"step{s}/query_logits"] = trainer.logits_expert_is_high(s_th, a_th, ns_th, d_th, logp).numpy()
            out[f"step{s}/query_logp"] = logp.numpy()
    out["stats_keys"] = np.array(sorted(stats))
    out["policy_M"] = policy.M.numpy()
    np.savez_compressed(os.path.join(OUT, name + ".npz"), **out)
    print("wrote", name, "final loss", stats["disc_loss"])


def running_norm_case():
    th.manual_seed(3)
    rn = ref_networks.RunningNorm(5)
    rn.train()
    out = {}
    for i, n in enumerate([1, 7, 64, 3]):
        x = th.randn(n, 5) * (i + 1) + i
        y = rn(x)
        out[f"x{i}"] = x.numpy()
        out[f"y{i}"] = y.numpy()
        out.update(_flat(f"s{i}", _state(rn)))
    rn.eval()
    x = th.randn(9, 5)
    out["x_eval"], out["y_eval"] = x.numpy(), rn(x).numpy()
    np.savez_compressed(os.path.join(OUT, "running_norm.npz"), **out)
    print("wrote running_norm")


def buffer_case():
    np.random.seed(11)
    rng = np.random.default_rng(11)
    buf = ref_buffer.ReplayBuffer(10, obs_shape=(3,), act_shape=(2,), obs_dtype=np.float32, act_dtype=np.float32)
    out = {}
    for i, n in enumerate([4, 5, 3, 17, 2]):
        t = _rand_transitions(rng, n, 3, 2)
        buf.store(ref_types.Transitions(infos=np.array([{}] * n), **t))
        out.update(_flat(f"store{i}", t))
        out[f"store{i}/idx"] = np.array([buf._buffer._idx, buf._buffer._n_data])
        out[f"store{i}/obs_arr"] = buf._buffer._arrays["obs"].copy()
        out[f"store{i}/dones_arr"] = buf._buffer._arrays["dones"].copy()
        s = buf.sample(6)
        out[f"sample{i}/obs"] = s.obs
        out[f"sample{i}/acts"] = s.acts
        out[f"sample{i}/dones"] = s.dones
    np.random.seed(5)
    out["randint_512_x8192"] = np.random.randint(512, size=8192)
    np.savez_compressed(os.path.join(OUT, "replay_buffer.npz"), **out)
    print("wrote replay_buffer")


def rollout_case():
    """BufferingWrapper -> pop -> flatten -> ReplayBuffer ordering, crossing an episode end."""
    out = {}
    for name, (E, T, H, cap, discrete) in dict(a=(3, 7, 5, 9, False), b=(4, 6, 50, 100, False),
                                               c=(5, 8, 4, 16, True)).items():
        spec = synth_env.SynthEnvSpec(4, 2, discrete=discrete, horizon=H, seed=7)
        venv = _HostVenv(synth_env.SynthVecEnv(spec, E, spaces_mod=spaces))
        bw = ref_wrappers.BufferingWrapper(venv)
        rng = np.random.default_rng(2)
        obs = bw.reset()
        acts_all = []
        for rnd in range(2):
            for t in range(T):
                a = rng.integers(0, 2, E) if discrete else rng.uniform(-1.5, 1.5, (E, 2)).astype(np.float32)
                acts_all.append(a)
                bw.step_async(a)
                bw.step_wait()
            trajs, ep_lens = bw.pop_trajectories()
            tr = ref_rollout.flatten_trajectories_with_rew(trajs)
            for k in ("obs", "acts", "next_obs", "dones", "rews"):
                out[f"{name}/round{rnd}/{k}"] = getattr(tr, k)
            out[f"{name}/round{rnd}/ep_lens"] = np.array(ep_lens)
            rb = ref_buffer.ReplayBuffer(cap, venv)
            rb.store(tr)
            out[f"{name}/round{rnd}/ring_obs"] = rb._buffer._arrays["obs"].copy()
            out[f"{name}/round{rnd}/ring_idx"] = np.array([rb._buffer._idx, rb._buffer._n_data])
        out[f"{name}/acts_fed"] = np.stack(acts_all)
        out[f"{name}/cfg"] = np.array([E, T, H, cap, int(discrete)])
    np.savez_compressed(os.path.join(OUT, "rollout_order.npz"), **out)
    print("wrote rollout_order")


def relabel_case():
    """RewardVecEnvWrapper(BufferingWrapper(venv)) with NormalizedRewardNet(BasicShapedRewardNet)."""
    th.manual_seed(4)
    E, T, H = 6, 9, 4
    spec = synth_env.SynthEnvSpec(5, 3, horizon=H, seed=9)
    venv = _HostVenv(synth_env.SynthVecEnv(spec, E, spaces_mod=spaces))
    net = ref_nets.BasicShapedRewardNet(venv.observation_space, venv.action_space,
                                        normalize_input_layer=ref_networks.RunningNorm)
    with ref_networks.training(net):  # give the input norms non-trivial stats
        net(th.randn(40, 5) * 2 + 1, th.randn(40, 3), th.randn(40, 5), th.zeros(40))
    nnet = ref_nets.NormalizedRewardNet(net, ref_networks.RunningNorm)
    bw = ref_wrappers.BufferingWrapper(venv)
    wrapped = ref_rw.RewardVecEnvWrapper(bw, nnet.predict_processed)
    rng = np.random.default_rng(8)
    out = _flat("net", _state(nnet))
    acts, rews, obs_l, dones_l = [], [], [], []
    for t in range(T):
        a = rng.uniform(-1.2, 1.2, (E, 3)).astype(np.float32)
        o, r, d, infos = wrapped.step(a)
        acts.append(a), rews.append(r), obs_l.append(o), dones_l.append(d)
    out.update(acts=np.stack(acts), rews=np.stack(rews), obs=np.stack(obs_l), dones=np.stack(dones_l))
    out.update(_flat("net_after", _state(nnet)))
    out["cfg"] = np.array([E, T, H])
    np.savez_compressed(os.path.join(OUT, "reward_relabel.npz"), **out)
    print("wrote reward_relabel")


def expert_loader_case():
    out = {}
    for seed, (n, B) in enumerate([(100, 32), (64, 64), (1000, 7)]):
        th.manual_seed(seed)
        t = ref_types.Transitions(obs=np.arange(n, dtype=np.float32)[:, None], acts=np.arange(n, dtype=np.float32)[:, None],
                                  next_obs=np.zeros((n, 1), np.float32), dones=np.zeros(n, bool),
                                  infos=np.array([{}] * n))
        it = ref_util.endless_iter(ref_base.make_data_loader(t, B))
        idx = [next(it)["acts"].numpy()[:, 0].astype(np.int64) for _ in range(3 * (n // B) + 2)]
        out[f"case{seed}/idx"] = np.stack(idx)
        out[f"case{seed}/cfg"] = np.array([n, B, seed])
    np.savez_compressed(os.path.join(OUT, "expert_loader.npz"), **out)
    print("wrote expert_loader")


def train_stats_case():
    th.manual_seed(6)
    out = {}
    for i, n in enumerate([0, 1, 10, 40]):
        logits = th.randn(2 * n) * 2
        labels = th.cat([th.ones(n, dtype=th.long), th.zeros(n, dtype=th.long)])
        loss = th.rand(())
        st = ref_common.compute_train_stats(logits, labels, loss)
        out[f"c{i}/logits"], out[f"c{i}/labels"], out[f"c{i}/loss"] = logits.numpy(), labels.numpy(), loss.numpy()
        out[f"c{i}/stats"] = np.array([st[k] for k in sorted(st)])
    out["keys"] = np.array(sorted(st))
    np.savez_compressed(os.path.join(OUT, "train_stats.npz"), **out)
    print("wrote train_stats")


def preference_case():
    """algorithms/preference_comparisons.py: RandomFragmenter, SyntheticGatherer, PreferenceModel,
    CrossEntropyRewardLoss on seeded trajectories and a seeded BasicRewardNet (single network and 3-member ensemble)."""
    from imitation.algorithms import preference_comparisons as ref_pc

    Do, Da, L, P = 11, 3, 25, 12
    rng = np.random.default_rng(21)
    trajs = []
    for i in range(6):
        n = int(rng.integers(30, 60))
        trajs.append(ref_types.TrajectoryWithRew(
            obs=rng.standard_normal((n + 1, Do)).astype(np.float32), acts=rng.uniform(-1, 1, (n, Da)).astype(np.float32),
            infos=None, terminal=bool(i % 2), rews=(0.3 * rng.standard_normal(n)).astype(np.float32)))
    out = {"cfg": np.array([Do, Da, L, P])}
    for i, t in enumerate(trajs):
        out.update(_flat(f"traj{i}", dict(obs=t.obs, acts=t.acts, rews=t.rews, terminal=np.array(t.terminal))))
    log = ref_logger.configure(os.path.join("/tmp", "imb_golden_log_pref"), format_strs=[])
    frags = ref_pc.RandomFragmenter(rng=np.random.default_rng(3), warning_threshold=0, custom_logger=log)(trajs, L, P)
    for i, (a, b) in enumerate(frags):
        out.update(_flat(f"pair{i}/a", dict(obs=a.obs, acts=a.acts, rews=a.rews, terminal=np.array(a.terminal))))
        out.update(_flat(f"pair{i}/b", dict(obs=b.obs, acts=b.acts, rews=b.rews, terminal=np.array(b.terminal))))
    out["prefs_prob"] = ref_pc.SyntheticGatherer(sample=False, temperature=0.5, discount_factor=0.9,
                                                 custom_logger=log)(frags)
    out["prefs_sampled"] = ref_pc.SyntheticGatherer(sample=True, rng=np.random.default_rng(4), custom_logger=log)(frags)
    out["prefs_t0"] = ref_pc.SyntheticGatherer(sample=False, temperature=0, custom_logger=log)(frags)
    obs_space = spaces.Box(-np.inf, np.inf, (Do,), np.float32)
    act_space = spaces.Box(-1.0, 1.0, (Da,), np.float32)
    th.manual_seed(8)
    net = ref_nets.BasicRewardNet(obs_space, act_space, hid_sizes=(32, 32))
    out.update(_flat("net", _state(net)))
    pm = ref_pc.PreferenceModel(net, noise_prob=0.1, discount_factor=0.95)
    prefs = out["prefs_sampled"].astype(np.float32)
    res = ref_pc.CrossEntropyRewardLoss()(frags, prefs, pm)
    probs, gt_probs = pm(frags)
    out["probs"], out["gt_probs"] = probs.detach().numpy(), gt_probs.numpy()
    out["loss"] = res.loss.detach().numpy()
    out["accuracy"], out["gt_reward_loss"] = res.metrics["accuracy"].numpy(), res.metrics["gt_reward_loss"].numpy()
    net.zero_grad()
    res.loss.backward()
    out.update(_flat("grad", {k: p.grad.numpy().copy() for k, p in net.named_parameters()}))
    # three-member ensemble: probabilities of all members (no gradient path, as in the reference)
    th.manual_seed(9)
    members = [ref_nets.BasicRewardNet(obs_space, act_space, hid_sizes=(32, 32)) for _ in range(3)]
    ens = ref_nets.RewardEnsemble(obs_space, act_space, members)
    for i, m in enumerate(members):
        out.update(_flat(f"member{i}", _state(m)))
    pme = ref_pc.PreferenceModel(ens, discount_factor=1.0)
    # (the reference's PreferenceModel.forward cannot hold per-member probabilities -- its `probs` buffer is 1-D --
    #  so the ensemble path is pinned through rewards() + probability(), the calls ActiveSelectionFragmenter makes)
    pe = [pme.probability(pme.rewards(ref_rollout.flatten_trajectories([a])),
                          pme.rewards(ref_rollout.flatten_trajectories([b]))) for a, b in frags]
    out["ensemble_probs"] = th.stack(pe).detach().numpy()
    # one BasicRewardTrainer epoch (AdamW, batch 8, minibatch 4) from the single network's initial weights
    th.manual_seed(10)
    ds = ref_pc.PreferenceDataset()
    ds.push(frags, prefs)
    trainer = ref_pc.BasicRewardTrainer(pm, ref_pc.CrossEntropyRewardLoss(), rng=np.random.default_rng(5), batch_size=8,
                                        minibatch_size=4, epochs=2, lr=1e-3, custom_logger=log)
    trainer.train(ds)
    out.update(_flat("net_trained", _state(net)))
    np.savez_compressed(os.path.join(OUT, "preference.npz"), **out)
    print("wrote preference")


def reference_api_case():
    """Host-side API of the reference on seeded inputs, for tests/test_oracle_vs_reference.py: data/serialize.py's
    demonstration directories, data/rollout.py helpers, algorithms/base.py's fixed-horizon check, data/types.py
    validation messages, preference_comparisons.py schedules / datasets / PreferenceModel, util/util.py oric and
    make_seeds, reward_nets.py preprocess and the reward registry, util/networks.py RunningNorm.
    Arrays go to reference_api.npz; everything else as one JSON document under its `facts` key."""
    import json
    import shutil

    from imitation.algorithms import preference_comparisons as ref_pc
    from imitation.data import serialize as ref_serialize
    from imitation.rewards import serialize as ref_ser

    out, facts = {}, {}
    # demonstration directories written by the reference (data/serialize.py:15-24)
    rng = np.random.default_rng(3)
    for discrete in (False, True):
        path = os.path.join(OUT, f"hf_reference_{int(discrete)}")
        shutil.rmtree(path, ignore_errors=True)
        ref_serialize.save(path, make_hf_trajectories(ref_types, rng, discrete))
    # rollout helpers (data/rollout.py:193-286, 509-621, 728-745)
    rng = np.random.default_rng(5)
    for monitor in (False, True):
        trajs = make_rollout_trajectories(ref_types, rng, monitor)
        facts[f"rollout_stats/{int(monitor)}"] = ref_rollout.rollout_stats(trajs)
        flat = ref_rollout.flatten_trajectories_with_rew(trajs)
        for field in ("obs", "acts", "next_obs", "dones", "rews"):
            out[f"flatten/{int(monitor)}/{field}"] = getattr(flat, field)
        facts[f"sample_until/{int(monitor)}"] = [bool(ref_rollout.make_sample_until(**kw)(trajs)) for kw in SAMPLE_UNTIL]
    facts["sample_until_errors"] = [error(lambda: ref_rollout.make_sample_until(**kw)) for kw in SAMPLE_UNTIL_BAD]
    arr = rng.standard_normal((7, 3))
    out["discounted_sum/input"] = arr
    for gamma in (1.0, 0.9):
        out[f"discounted_sum/{gamma}/2d"] = ref_rollout.discounted_sum(arr, gamma)
        out[f"discounted_sum/{gamma}/1d"] = ref_rollout.discounted_sum(arr[:, 0], gamma)
    # fixed-horizon check (algorithms/base.py:69-108): per step ["ok", remembered horizon] or ["err", message]
    for allow in (False, True):
        runs = []
        for script in HORIZON_SCRIPTS:
            algo, events = ref_base.BaseImitationAlgorithm(allow_variable_horizon=allow), []
            for horizons in script:
                try:
                    algo._check_fixed_horizon(horizons)
                except ValueError as e:
                    events.append(["err", str(e)])
                    break
                events.append(["ok", algo._horizon])
            runs.append(events)
        facts[f"fixed_horizon/{int(allow)}"] = runs
    # validation messages (data/types.py:61-330)
    cases, ok = validation_cases()
    facts["validation"] = {name: error(lambda: getattr(ref_types, cls)(**kw)) for name, (cls, kw) in cases.items()}
    facts["transitions_len"] = len(ref_types.Transitions(**ok))
    # comparison schedule (util.oric, make_seeds, QUERY_SCHEDULES; preference_comparisons.py:1465-1479, 1622-1636)
    rng = np.random.default_rng(0)
    oric = []
    for _ in range(500):
        n, total = int(rng.integers(1, 12)), int(rng.integers(0, 300))
        v = rng.random(n) + 1e-3
        oric.append(ref_util.oric(v / v.sum() * total).tolist())
    facts["oric"] = oric
    facts["make_seeds"] = [ref_util.make_seeds(np.random.default_rng(9), n) for n in (None, 1, 5)]
    facts["query_schedules"] = {name: [fn(t) for t in np.linspace(0, 1, 7)] for name, fn in ref_pc.QUERY_SCHEDULES.items()}
    facts["schedule_runs"] = {}
    for name, fn in ref_pc.QUERY_SCHEDULES.items():
        for total, iters, frac in SCHEDULE_RUNS:
            initial = int(total * frac)
            vec = np.array([fn(t) for t in np.linspace(0, 1, iters)])
            facts["schedule_runs"][f"{name}/{total}/{iters}/{frac}"] = \
                [initial] + ref_util.oric(vec / vec.sum() * (total - initial)).tolist()
    # RewardNet.preprocess and the reward-loader registry (reward_nets.py:74-118, rewards/serialize.py:230-260)
    facts["reward_registry"] = sorted(ref_ser.reward_registry.keys())
    rng = np.random.default_rng(0)
    for discrete in (True, False):
        net = ref_nets.BasicRewardNet(spaces.Box(-1, 1, (4,)), spaces.Discrete(3) if discrete else spaces.Box(-1, 1, (2,)))
        obs, nobs = rng.standard_normal((6, 4)), rng.standard_normal((6, 4)).astype(np.float32)
        acts = rng.integers(0, 3, 6) if discrete else rng.uniform(-1, 1, (6, 2))
        done = rng.random(6) < 0.5
        pre = net.preprocess(obs, acts, nobs, done)
        facts[f"preprocess/{int(discrete)}/dtypes"] = [str(t.dtype) for t in pre]
        for i, t in enumerate(pre):
            out[f"preprocess/{int(discrete)}/{i}"] = t.numpy()
        facts[f"state_dict_shapes/{int(discrete)}"] = {k: list(v.shape) for k, v in net.state_dict().items()}
    # TrajectoryDataset.sample / PreferenceDataset (preference_comparisons.py:99-124, 909-997)
    trajs = make_dataset_trajectories(ref_types)
    tds = ref_pc.TrajectoryDataset(trajs, np.random.default_rng(7))
    for steps in (10, 25, 46, 1):
        sample = tds.sample(steps)
        facts[f"trajectory_sample/{steps}/lens"] = [len(t) for t in sample]
        out[f"trajectory_sample/{steps}/obs"] = np.concatenate([t.obs for t in sample])
    facts["trajectory_sample_error"] = error(lambda: tds.sample(100), RuntimeError)
    pds = ref_pc.PreferenceDataset(max_size=3)
    f = trajs
    pds.push([(f[0], f[1]), (f[2], f[3])], np.array([1.0, 0.0], np.float32))
    pds.push([(f[4], f[5]), (f[6], f[0])], np.array([0.5, 1.0], np.float32))
    facts["preference_dataset_len"] = len(pds)
    out["preference_dataset/preferences"] = pds.preferences
    for i in range(3):
        (x, y), p = pds[i]
        out[f"preference_dataset/{i}/pref"], out[f"preference_dataset/{i}/x_obs"] = np.asarray(p), x.obs
        out[f"preference_dataset/{i}/y_acts"] = y.acts
    facts["preference_dataset_errors"] = [error(lambda: pds.push([(f[0], f[1]), (f[2], f[3])], bad))
                                          for bad in (np.array([1.0], np.float32), np.array([1.0, 0.0], np.float64))]
    # RunningNorm over training batches, then in eval mode (util/networks.py:19-134)
    norm = ref_networks.RunningNorm(5)
    g = th.Generator().manual_seed(0)
    for step in range(5):
        y = norm(th.randn(7 + step, 5, generator=g) * (1 + step) + step)
        out[f"running_norm/{step}/y"] = y.numpy()
        out.update(_flat(f"running_norm/{step}/state", _state(norm)))
    norm.eval()
    out["running_norm/eval/y"] = norm(th.randn(3, 5, generator=g)).numpy()
    out.update(_flat("running_norm/eval/state", _state(norm)))
    facts["running_norm_dtypes"] = {k: str(v.dtype) for k, v in norm.state_dict().items()}
    # PreferenceModel.probability and the cross-entropy loss (preference_comparisons.py:487-530, 1043-1090)
    net = ref_nets.BasicRewardNet(spaces.Box(-1, 1, (4,)), spaces.Box(-1, 1, (2,)))
    g = th.Generator().manual_seed(0)
    for i, (noise, discount, threshold) in enumerate(PREF_SETTINGS):
        pm = ref_pc.PreferenceModel(net, noise_prob=noise, discount_factor=discount, threshold=threshold)
        for scale in (0.3, 3.0):
            r1, r2 = th.randn(12, generator=g) * scale, th.randn(12, generator=g) * scale
            out[f"probability/{i}/{scale}"] = pm.probability(r1, r2).numpy()
        R1, R2 = th.randn(9, 12, generator=g) * 2, th.randn(9, 12, generator=g) * 2
        single = th.stack([pm.probability(x, y) for x, y in zip(R1, R2)])
        prefs = (th.rand(9, generator=g) < 0.5).float()
        out[f"probability/{i}/pairs"] = single.numpy()
        out[f"probability/{i}/bce"] = th.nn.functional.binary_cross_entropy(single, prefs).numpy()
        out[f"probability/{i}/accuracy"] = ((single > 0.5) == (prefs > 0.5)).float().mean().numpy()
    out["facts"] = np.array(json.dumps(facts, sort_keys=True))
    np.savez_compressed(os.path.join(OUT, "reference_api.npz"), **out)
    print("wrote reference_api")


def all_cases():
    """Every golden file of tests/golden/, (name, thunk) in generation order (shared with
    tests/test_oracle_vs_reference.py, which regenerates ALL of them from the reference)."""
    RN = ref_networks.RunningNorm
    return [
        ("disc_gail_hc", lambda: disc_case("disc_gail_hc", "gail", 17, 6, False, dict(normalize_input_layer=RN), 64, 64, 4, 0)),
        ("disc_gail_hc_minibatch", lambda: disc_case("disc_gail_hc_minibatch", "gail", 17, 6, False,
                                                     dict(normalize_input_layer=RN), 64, 16, 3, 1)),
        ("disc_gail_nonorm", lambda: disc_case("disc_gail_nonorm", "gail", 11, 3, False, dict(hid_sizes=(32,)), 32, 32, 3, 2)),
        ("disc_gail_cartpole", lambda: disc_case("disc_gail_cartpole", "gail", 4, 2, True, dict(hid_sizes=(64, 64)), 32, 32, 3, 3)),
        ("disc_gail_allinputs", lambda: disc_case("disc_gail_allinputs", "gail", 5, 2, False,
                                                  dict(use_next_state=True, use_done=True, normalize_input_layer=RN), 16, 8, 3, 4)),
        ("disc_airl_hc", lambda: disc_case("disc_airl_hc", "airl", 17, 6, False, dict(normalize_input_layer=RN), 64, 32, 4, 5,
                                           shaped=True)),
        ("disc_airl_nonorm", lambda: disc_case("disc_airl_nonorm", "airl", 6, 2, False,
                                               dict(reward_hid_sizes=(32, 32), potential_hid_sizes=(32,)), 16, 16, 3, 6,
                                               shaped=True)),
        ("running_norm", running_norm_case),
        ("replay_buffer", buffer_case),
        ("rollout_order", rollout_case),
        ("reward_relabel", relabel_case),
        ("expert_loader", expert_loader_case),
        ("train_stats", train_stats_case),
        ("preference", preference_case),
        ("reference_api", reference_api_case),
    ]


if __name__ == "__main__":
    os.makedirs(OUT, exist_ok=True)
    if len(sys.argv) > 1 and sys.argv[1] == "preference":
        preference_case()
        sys.exit(0)
    for _name, _thunk in all_cases():
        _thunk()
