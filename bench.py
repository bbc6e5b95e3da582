#!/usr/bin/env python
"""bench.py -- env-steps/sec of the adversarial-imitation round (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W [--impl ours|reference] [--config hc|cartpole|airl_hc|ant|pref]
                    [--dump-outputs DIR]

A "step" is one ROUND of the reference's hot path (AdversarialTrainer.train body, algorithms/adversarial/common.py:453-461):
generator rollout of E*T env steps with learned-reward relabel -> PPO update (n_epochs x minibatches) -> replay store ->
n_disc discriminator updates.  Default workload `hc` = the configuration BASELINE.json's metric is quoted on: GAIL on the
synthetic HalfCheetah-shaped env (obs 17 / act 6, horizon 1000) with the hyper-parameters of
scripts/config/tuned_hps/gail_seals_half_cheetah_best_hp_eval.json, E = 1024 envs per GPU (n_steps = 4096 / 1024 = 4), weak
scaling: every extra GPU adds 1024 envs.  The other BASELINE configs are selectable with --config (`pref` = reward-model
training of preference comparisons, a different unit: fragment-pair evaluations / s).

value   whole-job env-steps/s with everything resident in HBM (the captured-graph round): K timed rounds, split into up to
        --windows windows; the median of the windows' per-round times.
e2e     the same metric through the reference-facing API with HOST expert batches: every train_disc() gets `expert_samples`
        from pinned host memory (H2D inside the timed region) and returns its Mapping[str, float] (D2H inside the timed region);
        K timed rounds in up to 3 windows.
--dump-outputs DIR  after the K timed captured-graph rounds, write what the last one left to its caller as DIR/<name>.npy
        (float32 / float64): the round's discriminator statistics [n_disc, 16] and the trained policy and reward network
        (state_dict entries).  Seeds are fixed, so two builds run with the same arguments can be compared output for output.
roofline  dominant kernel by time share (the persistent PPO update); `roofline_disc`: the tcgen05 discriminator kernel on a
        2^20-row sweep point (tensor-pipe % from the committed ncu capture); `roofline_stages`: achieved GB/s of the stage-1/2
        kernels (rollout, sample+gather, ring store), all against MEASURED_PEAKS.json.
cpu_baseline / --impl reference  the CPU restatement of the reference's loop (oracle/gail_port.py: reference data plane +
        SB3-PPO restatement, torch-CPU eager) on this box's host cores, with a per-stage table.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np
import torch as th

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # the tree may be read-only: leave no __pycache__ in it

# Per-GPU sizes (weak scaling).  `ppo`: SB3 PPO keyword arguments of the tuned JSON / script defaults.
CONFIGS = {
    "hc": dict(
        title="GAIL HalfCheetah-shaped synthetic env (obs17/act6, H=1000), tuned HPs gail_seals_half_cheetah_best_hp_eval.json: "
              "demo_batch 8192, replay 512, 8 disc updates/round, PPO batch 4096 / mb 64 / 5 epochs; BasicRewardNet 32x32 + "
              "RunningNorm; FeedForward32Policy + NormalizeFeaturesExtractor",
        algo="gail", d_obs=17, d_act=6, discrete=False, horizon=1000, envs_per_gpu=1024, ppo_batch=4096, ppo_minibatch=64,
        ppo_epochs=5, demo_batch=8192, replay_capacity=512, n_disc=8, hid=(32, 32), norm_features=True,
        ppo=dict(clip_range=0.1, ent_coef=3.992371122209408e-6, gae_lambda=0.95, gamma=0.95,
                 learning_rate=0.00026250519057717037, max_grad_norm=0.8, vf_coef=0.11483689492120866)),
    "cartpole": dict(
        title="GAIL seals/CartPole-shaped synthetic env (obs4 / Discrete(2), H=500), script defaults "
              "(scripts/config/train_adversarial.py:27-51, ingredients/rl.py:59-66): demo_batch 1024, 4 disc updates/round, "
              "replay = PPO batch 2048 / mb 64 / 10 epochs, 64 envs; BasicRewardNet 64x64 + RunningNorm; FeedForward32Policy",
        algo="gail", d_obs=4, d_act=2, discrete=True, horizon=500, envs_per_gpu=64, ppo_batch=2048, ppo_minibatch=64,
        ppo_epochs=10, demo_batch=1024, replay_capacity=2048, n_disc=4, hid=(64, 64), norm_features=False,
        ppo=dict(learning_rate=3e-4, ent_coef=0.0)),
    "airl_hc": dict(
        title="AIRL HalfCheetah-shaped synthetic env (obs17/act6, H=1000), tuned HPs airl_seals_half_cheetah_best_hp_eval.json: "
              "demo_batch 2048, replay 512, 16 disc updates/round, PPO batch 8192 / mb 64 / 5 epochs; BasicShapedRewardNet "
              "(base 23->32->1, potential 17->32->32->1) + RunningNorm in and out; FeedForward32Policy + NormalizeFeaturesExtractor",
        algo="airl", d_obs=17, d_act=6, discrete=False, horizon=1000, envs_per_gpu=1024, ppo_batch=8192, ppo_minibatch=64,
        ppo_epochs=5, demo_batch=2048, replay_capacity=512, n_disc=16, hid=(32,), norm_features=True,
        ppo=dict(clip_range=0.1, ent_coef=0.0005544771755195421, gae_lambda=0.95, gamma=0.95,
                 learning_rate=0.00047248619386801587, max_grad_norm=0.8, vf_coef=0.11483689492120866)),
    "ant": dict(
        title="GAIL Ant-shaped synthetic env (obs27/act8, H=1000), tuned HPs gail_seals_ant_best_hp_eval.json scaled per GPU of "
              "an 8-GPU job (4096 envs / 8 = 512 envs, PPO batch 16384 / 8 = 2048, replay 16384 / 8 = 2048): demo_batch 32, "
              "8 disc updates/round, PPO mb 16 / 10 epochs; BasicRewardNet 32x32 + RunningNorm; FeedForward32Policy + "
              "NormalizeFeaturesExtractor",
        algo="gail", d_obs=27, d_act=8, discrete=False, horizon=1000, envs_per_gpu=512, ppo_batch=2048, ppo_minibatch=16,
        ppo_epochs=10, demo_batch=32, replay_capacity=2048, n_disc=8, hid=(32, 32), norm_features=True,
        ppo=dict(clip_range=0.3, ent_coef=0.008871887607426377, gae_lambda=0.8, gamma=0.995,
                 learning_rate=2.428297806883194e-05, max_grad_norm=0.9, vf_coef=0.4351450387648799)),
}
for _c in CONFIGS.values():
    _c.setdefault("n_expert_episodes", 60)
    _c.setdefault("seed", 0)

PPO_DRAM_BYTES_NCU = 611584 + 0        # bytes per launch, profiles/ncu_ppo_r02c_selected.csv (read + write), hc config
DISC_TC_NCU = dict(source="profiles/ncu_disc_tc_r02_selected.csv (k_disc_fwdbwd_tc<8>, 2^20 rows, --set full)",
                   dram_bytes=96830208 + 4711424, tensor_pipe_pct_of_elapsed=37.4, issue_active_pct=53.4)


# -------------------------------------------------------------------------------------------------
def synth_expert(env_params: np.ndarray, d_obs, d_act, horizon, n_episodes, seed, discrete=False):
    """Synthetic expert: fixed random linear-tanh policy + small noise, rolled out in the env."""
    rng = np.random.default_rng(seed + 1000)
    A = env_params[:d_obs * d_obs].reshape(d_obs, d_obs)
    Bm = env_params[d_obs * d_obs:d_obs * d_obs + d_obs * d_act].reshape(d_obs, d_act)
    c = env_params[d_obs * d_obs + d_obs * d_act:d_obs * d_obs + d_obs * d_act + d_obs]
    K = rng.standard_normal((d_act, d_obs)).astype(np.float32) * 0.7
    obs = (0.1 * rng.standard_normal((n_episodes, d_obs))).astype(np.float32)
    O, Ac, NO, D = [], [], [], []
    for t in range(horizon):
        act = np.tanh(obs @ K.T) + 0.1 * rng.standard_normal((n_episodes, d_act)).astype(np.float32)
        if discrete:
            a = act.argmax(1)
            u = np.eye(d_act, dtype=np.float32)[a]
            Ac.append(a.astype(np.int64))
        else:
            u = np.clip(act, -1, 1).astype(np.float32)
            Ac.append(u)
        nobs = np.tanh(obs @ A.T + u @ Bm.T + c).astype(np.float32)
        O.append(obs), NO.append(nobs), D.append(np.full(n_episodes, t == horizon - 1))
        obs = nobs
    # episode-major order like flatten_trajectories
    sw = lambda x: np.ascontiguousarray(np.swapaxes(np.stack(x), 0, 1)).reshape(n_episodes * horizon, *x[0].shape[1:])
    return dict(obs=sw(O), acts=sw(Ac), next_obs=sw(NO), dones=sw(D).astype(bool))


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""

    def __init__(self, index: int, enabled: bool = True):
        self.index, self.rows, self._stop, self.enabled = index, [], threading.Event(), enabled
        self.t = threading.Thread(target=self._run, daemon=True)

    def _run(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i",
                                      str(self.index)], capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            self._stop.wait(0.2)

    def __enter__(self):
        if self.enabled:
            self.t.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        if self.enabled:
            self.t.join(timeout=3)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        sm = sorted(float(r[0]) for r in self.rows if r[0].replace(".", "").isdigit())
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(r[3 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": float(self.rows[0][1]),
                "power_w_max": max(float(r[2]) for r in self.rows), "samples": len(self.rows), "reasons": reasons}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def pin_to_gpu_numa(local: int, n_local: int) -> str:
    """Restrict this rank to a private share of the host cores of ITS GPU's NUMA node (8 ranks x (python + torch threads +
    shuffle worker) on one box otherwise migrate across sockets; the per-step collectives serialise every rank's jitter)."""
    try:
        def node_of(i):
            p = th.cuda.get_device_properties(i)
            path = f"/sys/bus/pci/devices/{p.pci_domain_id:04x}:{p.pci_bus_id:02x}:{p.pci_device_id:02x}.0/numa_node"
            return max(0, int(open(path).read().strip()))

        def cpus_of(node):
            out = []
            for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
                a, _, b = part.partition("-")
                out += list(range(int(a), int(b or a) + 1))
            return out

        nodes = [node_of(i) for i in range(n_local)]
        mine = nodes[local]
        peers = [i for i in range(n_local) if nodes[i] == mine]
        allowed = sorted(set(cpus_of(mine)) & set(os.sched_getaffinity(0)))
        share = max(2, len(allowed) // len(peers))
        k = peers.index(local)
        cpus = allowed[k * share:(k + 1) * share] or allowed
        os.sched_setaffinity(0, cpus)
        return f"numa node {mine}, {len(cpus)} cores"
    except Exception as e:  # (containers without sysfs topology: leave the scheduler alone)
        return f"unpinned ({type(e).__name__})"


# -------------------------------------------------------------------------------------------------
# reference arm / cpu_baseline: the CPU restatement of the reference's loop
# -------------------------------------------------------------------------------------------------
def build_cpu_port(n_envs, cfg, env_id_offset=0):
    from oracle import gail_port, nets_port, ppo_port, synth_env

    th.manual_seed(cfg["seed"])
    np.random.seed(cfg["seed"])
    disc = cfg["discrete"]
    spec = synth_env.SynthEnvSpec(cfg["d_obs"], cfg["d_act"], discrete=disc, horizon=cfg["horizon"], seed=cfg["seed"])
    venv = synth_env.SynthVecEnv(spec, n_envs, env_id_offset=env_id_offset)
    env_params = np.concatenate([spec.A.ravel(), spec.Bm.ravel(), spec.c, spec.w])
    expert = synth_expert(env_params, cfg["d_obs"], cfg["d_act"], cfg["horizon"], cfg["n_expert_episodes"], cfg["seed"], disc)
    pol = ppo_port.ActorCriticPort(cfg["d_obs"], cfg["d_act"], discrete=disc, normalize_features=cfg["norm_features"])
    gen = ppo_port.PPOPort(pol, venv, n_steps=cfg["ppo_batch"] // n_envs, batch_size=cfg["ppo_minibatch"],
                           n_epochs=cfg["ppo_epochs"], **cfg["ppo"])
    if cfg["algo"] == "airl":
        net = nets_port.ShapedRewardNetPort(cfg["d_obs"], cfg["d_act"], reward_hid_sizes=cfg["hid"], normalize_input=True)
    else:
        net = nets_port.BasicRewardNetPort(cfg["d_obs"], cfg["d_act"], hid_sizes=cfg["hid"], normalize_input=True)
    tr = gail_port.AdversarialPort(venv=venv, expert=expert, demo_batch_size=cfg["demo_batch"], gen=gen,
                                   reward_net=net, airl=cfg["algo"] == "airl", normalize_output=cfg["algo"] == "airl",
                                   n_disc_updates_per_round=cfg["n_disc"],
                                   gen_replay_buffer_capacity=cfg["replay_capacity"])
    return tr


def pick_cpu_threads(cfg, n_envs):
    """The reference's tensors are tiny (MLPs of width 32, minibatches of 64): oversubscribing a
    many-core host makes torch-CPU *slower* (measured: 128 threads -> 87 s/round vs ~1 s/round at 8).
    Give the baseline the thread count it runs fastest with: time one PPO-minibatch-sized and one
    disc-batch-sized step at a few candidates and keep the best (the reference's own CI pins 1)."""
    import time as _t

    ncpu = os.cpu_count() or 1
    cands = sorted({c for c in (1, 2, 4, 8, 16, 32) if c <= ncpu})
    mlp = th.nn.Sequential(th.nn.Linear(23, 32), th.nn.ReLU(), th.nn.Linear(32, 32), th.nn.ReLU(), th.nn.Linear(32, 1))
    opt = th.optim.Adam(mlp.parameters())
    xs, xb = th.randn(cfg["ppo_minibatch"], 23), th.randn(2 * cfg["demo_batch"], 23)
    best, best_t = 1, float("inf")
    for c in cands:
        th.set_num_threads(c)
        t0 = _t.perf_counter()
        for x, reps in ((xs, 40), (xb, 2)):
            for _ in range(reps):
                opt.zero_grad()
                mlp(x).square().mean().backward()
                opt.step()
        dt = _t.perf_counter() - t0
        if dt < best_t:
            best, best_t = c, dt
    return best


def time_cpu_port(cfg, n_envs, steps, warmup, stages=False):
    """-> (env-steps/s, s per round, threads, {stage: ms per round}).  Stages = the rows of SURVEY 6 / BASELINE.md 3:
    rollout (policy + env + wrappers + relabel), PPO update, pop/flatten/store, the n_disc discriminator updates."""
    th.set_num_threads(pick_cpu_threads(cfg, n_envs))
    tr = build_cpu_port(n_envs, cfg)
    acc = {}

    def wrap(obj, name, label):
        fn = getattr(obj, name)

        def w(*a, **k):
            t0 = time.perf_counter()
            try:
                return fn(*a, **k)
            finally:
                acc[label] = acc.get(label, 0.0) + time.perf_counter() - t0
        setattr(obj, name, w)

    per = tr.gen_train_timesteps
    if warmup:
        tr.train(per * warmup)
    if stages:
        wrap(tr.gen, "collect_rollouts", "rollout: policy + env step + BufferingWrapper + reward relabel")
        wrap(tr.gen, "train", "PPO update (n_epochs x minibatches)")
        wrap(tr.buffering, "pop_trajectories", "pop_trajectories")
        wrap(tr.replay, "store", "ReplayBuffer.store")
        wrap(tr, "train_disc", "discriminator updates (sample + batch + fwd/BCE/bwd + Adam + stats)")
    t0 = time.perf_counter()
    tr.train(per * steps)
    dt = time.perf_counter() - t0
    table = {k: round(v / steps * 1e3, 3) for k, v in acc.items()}
    if stages:
        table["other (flatten, fixed-horizon check, loop)"] = round(max(0.0, dt - sum(acc.values())) / steps * 1e3, 3)
    return per * steps / dt, dt / steps, th.get_num_threads(), table


# -------------------------------------------------------------------------------------------------
# our arm
# -------------------------------------------------------------------------------------------------
def build_trainer(cfg, rank, world, device):
    from imitation_b200 import _desc
    from imitation_b200.algorithms import ppo
    from imitation_b200.algorithms.adversarial import airl, gail
    from imitation_b200.envs import synth
    from imitation_b200.rewards import reward_nets
    from imitation_b200.util import networks

    E = cfg["envs_per_gpu"]
    th.manual_seed(cfg["seed"])
    venv = synth.DeviceVecEnv(cfg["d_obs"], cfg["d_act"], E, discrete=cfg["discrete"], horizon=cfg["horizon"],
                              seed=cfg["seed"], env_id_offset=rank * E, device=device)
    expert = synth_expert(_desc.synth_env_params(cfg["d_obs"], cfg["d_act"], cfg["seed"]), cfg["d_obs"], cfg["d_act"],
                          cfg["horizon"], cfg["n_expert_episodes"], cfg["seed"], cfg["discrete"])
    gen = ppo.DevicePPO("FeedForward32Policy", venv, n_steps=cfg["ppo_batch"] // E, batch_size=cfg["ppo_minibatch"],
                        n_epochs=cfg["ppo_epochs"], policy_kwargs=dict(normalize_features=cfg["norm_features"]),
                        seed=cfg["seed"] + rank, device=device, **cfg["ppo"])
    if cfg["algo"] == "airl":
        net = reward_nets.BasicShapedRewardNet(venv.observation_space, venv.action_space, reward_hid_sizes=cfg["hid"],
                                               normalize_input_layer=networks.RunningNorm)
        net = reward_nets.NormalizedRewardNet(net, normalize_output_layer=networks.RunningNorm)
        cls = airl.AIRL
    else:
        net = reward_nets.BasicRewardNet(venv.observation_space, venv.action_space, hid_sizes=cfg["hid"],
                                         normalize_input_layer=networks.RunningNorm)
        cls = gail.GAIL
    tr = cls(demonstrations=expert, demo_batch_size=cfg["demo_batch"], venv=venv, gen_algo=gen, reward_net=net,
             n_disc_updates_per_round=cfg["n_disc"], gen_replay_buffer_capacity=cfg["replay_capacity"],
             sampling="device", seed=cfg["seed"] + 17 * rank)
    return tr, expert


def cuda_time_ms(fn):
    a, b = th.cuda.Event(enable_timing=True), th.cuda.Event(enable_timing=True)
    a.record()
    fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b)


def stage_rooflines(tr, cfg, peak):
    """Achieved GB/s of the stage-1/2 kernels at this configuration, each timed alone with CUDA events over 50 launches
    (algorithmic bytes = SURVEY 8(d) per-unit figures x units per launch).  They are latency-bound at the tuned sizes
    (a rollout moves ~1.3 MB, a gather ~2.7 MB): the fractions document that, they are not a target."""
    from imitation_b200 import _desc, _lib

    gen, v = tr.gen_algo, tr.venv
    E, T, Do, Da = v.num_envs, gen.n_steps, v.d_obs, v.d_act
    tw = _desc.table_width(Do, Da)
    out = {}
    reps = 50
    th.cuda.synchronize()

    def timed(fn):
        fn()
        th.cuda.synchronize()
        return cuda_time_ms(lambda: [fn() for _ in range(reps)]) / reps

    # rollout (k_rollout): per env step 4*(2 Do + Da) + 4 + 1 read/write of env state and record + the PPO row
    rw = _lib.rollout_row_width(gen.policy.desc)
    ms = timed(lambda: gen.collect_rollouts())  # rollout + GAE + counter advance (3 launches)
    b = E * T * (4 * (2 * Do + Da) + 5 + 4 * Do + 4 * rw + 4 * tw)
    out["collect_rollouts (k_rollout + k_gae + advance)"] = dict(ms=ms, bytes=b, GB_s=b / ms / 1e6, frac=b / ms / 1e6 / peak)
    tr.venv_buffering.discard()
    # sample + gather (k_sample_gather): idx + 4 tw read + 4 tw write per gathered row, 2 mb rows per launch
    B, mb = tr.demo_batch_size, tr.demo_minibatch_size
    ring = tr._gen_replay_buffer
    ms = timed(lambda: _lib.disc_sample_gather(tr._expert_table, tr._expert_n, ring.table, ring.capacity, tr._tw, mb, 0,
                                               tr.seed, tr._expert_state, tr.venv.state, tr._batch, tr._ld))
    b = 2 * mb * (8 + 8 * tw)
    out["k_sample_gather (index draw + expert|generator gather)"] = dict(ms=ms, bytes=b, GB_s=b / ms / 1e6,
                                                                        frac=b / ms / 1e6 / peak)
    # ring store (k_table_store): one round of generator samples packed into AoS rows
    n = E * T
    obs = th.randn(n, Do, device=v.device)
    acts = th.randn(n, Da, device=v.device)
    dones = th.zeros(n, dtype=th.uint8, device=v.device)
    table = th.zeros(max(n, 1), tw, device=v.device)
    st = th.zeros(_lib.ST_WORDS, dtype=th.int64, device=v.device)
    if v.discrete:
        ai = th.randint(0, Da, (n,), device=v.device)
        ms = timed(lambda: _lib.table_store(table, n, Do, Da, obs, None, ai, obs, dones, n, False, st))
    else:
        ms = timed(lambda: _lib.table_store(table, n, Do, Da, obs, acts, None, obs, dones, n, False, st))
    b = n * 2 * 4 * tw
    out["k_table_store (transitions -> AoS table rows)"] = dict(ms=ms, bytes=b, GB_s=b / ms / 1e6, frac=b / ms / 1e6 / peak)
    for d in out.values():
        for k in ("ms", "GB_s", "frac"):
            d[k] = round(d[k], 6)
    return out


def disc_roofline(tr, peak, device):
    """The fused discriminator fwd/BCE/bwd kernel at 2^20 rows (three rotating 96 MB input buffers defeat L2): the tcgen05
    path and, beside it, the fp32-FFMA kernel of round 1."""
    from imitation_b200 import _desc, _lib

    eng = tr._fused_net.engine()
    d = eng.desc
    if d.shaped or d.base.n_hidden != 2 or d.base.h1 != 32 or d.base.h2 != 32 or d.base.din > 31:
        return None  # (shapes outside the tensor-core kernel: the FFMA kernel's numbers are in profiles/)
    n_big = 1 << 20
    din = d.base.din
    ld = _desc.batch_ld(n_big)
    bufs = [th.randn(din, ld, device=device) for _ in range(3)]
    logits = th.empty(n_big, device=device)
    res = {}
    for name, fl in (("tc", 0), ("ffma", _lib.IMB_F_NO_TENSOR)):
        def run(i):
            _lib.disc_fwd_bwd(d, eng.params, eng.norm_state, bufs[i % 3], ld, n_big, n_big // 2, 1.0 / n_big, None, logits,
                              _lib.IMB_F_ZERO_GRAD | fl, eng.ws)
        for i in range(3):
            run(i)
        th.cuda.synchronize()
        reps = 9
        res[name] = cuda_time_ms(lambda: [run(i) for i in range(reps)]) / reps
    bpr = 4 * din + 4
    flop = 2 * (3 * (din * 32 + 32 * 32 + 32)) - 2 * din * 32
    ach = n_big * bpr / (res["tc"] / 1e3) / 1e9
    return {"kernel": "k_disc_fwdbwd_tc (tcgen05 3xTF32 split: fused BasicRewardNet fwd + BCE + bwd + weight gradients), "
                      f"2^20 rows, Din {din}, 32x32",
            "bound": "tensor", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
            "traffic": DISC_TC_NCU["dram_bytes"], "algorithmic_bytes_per_launch": n_big * bpr,
            "ms_per_launch": res["tc"], "Grows_per_s": n_big / (res["tc"] / 1e3) / 1e9,
            "fp32_equivalent_tflops": n_big * flop / (res["tc"] / 1e3) / 1e12,
            "tensor_pipe_pct_of_elapsed_ncu": DISC_TC_NCU["tensor_pipe_pct_of_elapsed"], "ncu_source": DISC_TC_NCU["source"],
            "ffma_kernel_ms_per_launch": res["ffma"], "speedup_vs_ffma_kernel": res["ffma"] / res["tc"],
            "note": "includes the gradient-accumulator memset node.  What binds: per 128-row tile the 3xTF32 contractions "
                    "cost 33 TS MMAs x 16 cycles + 48 SS MMAs x 30 cycles = 1968 tensor-pipe cycles (the weight-gradient MMAs "
                    "run at M=64 with half of each accumulator unused), i.e. a ceiling of 14.4 G rows/s = 21% of the HBM "
                    "roofline at 96 B/row; measured ~5.4 k cycles per tile: the chain of 4 epilogue phases and 3 "
                    "tensor-core hand-offs per tile is serial because only one set of weight-gradient operand tiles "
                    "(128 KB) fits in shared memory (profiles/r02_summary.md)"}


def split_rounds(k: int, windows: int) -> list:
    """k timed rounds over min(windows, k) windows of near-equal size."""
    n = max(1, min(windows, k))
    return [k // n + (i < k % n) for i in range(n)]


def dump_outputs(tr, round_stats, out_dir):
    """What one captured-graph round leaves to its caller: the round's discriminator statistics and the trained policy and
    reward network, as float32 / float64 .npy files (integer buffers as float64)."""
    os.makedirs(out_dir, exist_ok=True)
    arrays = {"round_stats": round_stats}
    for prefix, module in (("policy", tr.policy), ("reward_net", tr.reward_train)):
        arrays.update({f"{prefix}.{k}": v for k, v in module.state_dict().items()})
    for name, v in arrays.items():
        a = v.detach().cpu().numpy()
        np.save(os.path.join(out_dir, name + ".npy"), a if a.dtype in (np.float32, np.float64) else a.astype(np.float64))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200, help="timed rounds (each metric times this many)")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="hc", choices=sorted(CONFIGS) + ["pref"])
    ap.add_argument("--cpu-rounds", type=int, default=12, help="rounds of the CPU baseline sample (rank 0, N=1)")
    ap.add_argument("--host-threads", type=int, default=4,
                    help="torch intra-op threads for the host side of the loop (all its CPU ops are tiny; the default pool of one thread per core makes the DataLoader-style shuffle ~30x slower); 0: leave torch default")
    ap.add_argument("--windows", type=int, default=5,
                    help="windows the --steps timed rounds are split into; the median per-round time is reported")
    ap.add_argument("--no-pin", action="store_true", help="do not pin the rank to its GPU's NUMA node")
    ap.add_argument("--profile-host", action="store_true", help="wall-clock breakdown of the e2e loop (every rank -> stderr)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed round's outputs to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.config == "pref" or args.impl != "ours"):
        ap.error("--dump-outputs writes the outputs of the GPU adversarial round (--impl ours, not --config pref)")
    if args.config == "pref":
        import importlib.util

        spec = importlib.util.spec_from_file_location("pref_bench", os.path.join(ROOT, "profiles", "pref_bench.py"))
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
        args.hbm_peak, args.hbm_peak_source = peaks()
        return mod.main(args)
    cfg = CONFIGS[args.config]
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    E, T = cfg["envs_per_gpu"], cfg["ppo_batch"] // cfg["envs_per_gpu"]
    config = {"workload": cfg["title"], "name": args.config,
              "envs_per_gpu": E, "n_steps": T, "env_steps_per_round_per_gpu": E * T, "parallelism": f"dp{world}",
              "sync": "discriminator: global-batch step (all-gather of RunningNorm batch moments + all-reduce of [gradients | "
                      "statistic sums] per optimiser step, replicas bit-identical); generator: one all-reduce per round "
                      "(params + Adam moments averaged, RunningNorm merged exactly)",
              "streams": "GAIL: the discriminator updates run on a second stream beside the PPO update (independent given "
                         "the rollouts; bit-identical to the serial order); AIRL: one stream",
              "l2_policy": "the working set of a round (rollout table, ring, disc batch, expert table: a few MB) is L2-resident "
                           "by construction at the tuned sizes; the roofline sweep point uses 2^20 rows x 3 rotating buffers"}

    # ------------------------------------------------------------------------------ reference arm
    if args.impl == "reference":
        if rank != 0:
            return
        steps, warmup = max(1, args.steps), max(0, args.warmup)
        v, spr, cores, table = time_cpu_port(cfg, E, steps, warmup, stages=True)
        line = {"impl": "reference", "metric": "GAIL env-steps/sec (disc+gen loop)", "value": v, "unit": "env-steps/s",
                "n_gpus": args.gpus, "steps": steps, "warmup": warmup, "ms_per_step": spr * 1e3,
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": config,
                "cpu_baseline": {"value": v, "unit": "env-steps/s", "cores": cores, "kind": "port",
                                 "stages_ms_per_round": table,
                                 "sample": f"{steps} rounds of {E * T} env steps (E={E} envs on one host process; "
                                           "oracle/gail_port.py = reference data plane + SB3-PPO restatement, torch-CPU; "
                                           f"torch threads auto-picked = {cores} of {os.cpu_count()} host cores, the "
                                           "fastest setting for these tiny tensors)"},
                "e2e": {"value": v, "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line))
        return

    # ------------------------------------------------------------------------------ our arm
    import torch.distributed as dist

    n_local = int(os.environ.get("LOCAL_WORLD_SIZE", str(world)))
    th.cuda.set_device(local)
    device = th.device("cuda", local)
    affinity = "not pinned (--no-pin)" if args.no_pin else pin_to_gpu_numa(local, n_local)
    if args.host_threads > 0:
        th.set_num_threads(args.host_threads)  # torch CPU ops on the host side of the loop are all tiny
    config["host"] = f"rank affinity: {affinity}; torch threads {th.get_num_threads()}"
    if world > 1:
        dist.init_process_group("nccl", device_id=device)
    from imitation_b200 import _lib, distributed

    tr, expert = build_trainer(cfg, rank, world, device)
    sync = None
    if world > 1:
        if cfg["algo"] == "gail":
            tr.set_distributed()  # global-batch discriminator steps
        sync = distributed.trainer_round_sync(tr)
        sync.broadcast_initial(0)

    def round_eager():
        if sync:
            sync.begin_round()
        tr.train_gen()
        tr.disc_train_mode = True
        for _ in range(cfg["n_disc"]):
            tr.train_disc_async(check_ring=False)
        tr.disc_train_mode = False
        tr.join()  # (the discriminator updates run on their own stream beside the PPO update)
        if sync:
            sync.end_round()

    def round_graph():
        if sync:
            sync.begin_round()
        tr.replay_round()
        if sync:
            sync.end_round()

    # warm-up: exactly W rounds (at least 3): two eager ones (allocations, function attributes, the rollout graphs), the
    # capture (no work executed), the rest as replays of the captured round
    W = max(3, args.warmup)
    for _ in range(2):
        round_eager()
    th.cuda.synchronize()
    tr.capture_round()
    for _ in range(W - 2):
        round_graph()
    th.cuda.synchronize()

    # ---- value: K graph-replayed rounds in windows, device timed, max over ranks, median per-round time over windows ----
    K = args.steps
    win_ms, win_rounds, launches = [], split_rounds(K, args.windows), 0
    with ClockSampler(local, enabled=(rank == 0)) as clocks:
        for k in win_rounds:
            if world > 1:
                dist.barrier()
            th.cuda.synchronize()
            l0 = _lib.LAUNCHES["count"]
            ms = cuda_time_ms(lambda: [round_graph() for _ in range(k)])
            launches += _lib.LAUNCHES["count"] - l0
            th.cuda.synchronize()
            if world > 1:
                t = th.tensor([ms], device=device)
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                ms = float(t)
            win_ms.append(ms)
        if world > 1:
            dist.barrier()
    ms_round = statistics.median(m / k for m, k in zip(win_ms, win_rounds))
    value = world * E * T / (ms_round / 1e3)
    if args.dump_outputs and rank == 0:
        dump_outputs(tr, tr._round_stats, args.dump_outputs)

    # ---- e2e: reference-facing API, host expert batches, stats read back every update ---------------------------
    # Host side = what a DataLoader(shuffle=True, drop_last=True) does: the demonstrations live in pinned
    # host memory, are re-shuffled once per epoch (timed) and handed to train_disc() as contiguous batches;
    # every train_disc() copies its batch H2D and returns Mapping[str, float] (one D2H read).
    B = cfg["demo_batch"]
    n_exp = len(expert["obs"])

    def host_t(v):
        if v.dtype == bool:
            return th.as_tensor(np.ascontiguousarray(v))
        if np.issubdtype(v.dtype, np.integer):
            return th.as_tensor(np.ascontiguousarray(v.astype(np.int64)))
        return th.as_tensor(np.ascontiguousarray(v.astype(np.float32)))

    src = {k: host_t(v) for k, v in expert.items()}
    # two pinned epoch buffers; the NEXT epoch is shuffled by a worker thread (what DataLoader workers do)
    bufs = [{k: th.empty_like(v).pin_memory() for k, v in src.items()} for _ in range(2)]
    host_gen = th.Generator().manual_seed(1234 + rank)
    import concurrent.futures

    pool = concurrent.futures.ThreadPoolExecutor(max_workers=1)

    def shuffle_into(buf):
        perm = th.randperm(n_exp, generator=host_gen)
        for k in src:
            th.index_select(src[k], 0, perm, out=buf[k])
        return buf

    ep_state = {"pos": 0, "cur": shuffle_into(bufs[0]), "next": pool.submit(shuffle_into, bufs[1]), "i": 0}
    shuffled = ep_state["cur"]

    def next_host_batch():
        if ep_state["pos"] + B > n_exp:  # drop_last, new epoch
            ep_state["cur"] = ep_state["next"].result()
            ep_state["i"] ^= 1
            ep_state["next"] = pool.submit(shuffle_into, bufs[ep_state["i"] ^ 1])
            ep_state["pos"] = 0
        lo = ep_state["pos"]
        ep_state["pos"] = lo + B
        return {k: v[lo:lo + B] for k, v in ep_state["cur"].items()}

    h2d = cfg["n_disc"] * sum(v[:B].numel() * v.element_size() for v in shuffled.values())
    d2h = cfg["n_disc"] * 9 * 4
    from imitation_b200.util import networks

    def round_e2e():
        if sync:
            sync.begin_round()
        tr.train_gen()
        for _ in range(cfg["n_disc"]):
            with networks.training(tr.reward_train):
                tr.train_disc(expert_samples=next_host_batch())  # H2D copy + update + 9-float D2H
        if sync:
            tr.join()
            sync.end_round()

    for _ in range(3):
        round_e2e()
    th.cuda.synchronize()
    if world > 1:
        dist.barrier()
    if args.profile_host:
        # wall-clock breakdown of the e2e loop on EVERY rank (cProfile's per-call overhead distorts this loop badly)
        acc = {}

        def wrap(obj, name, label=None):
            fn = getattr(obj, name)
            lab = label or name

            def w(*a, **k):
                t0 = time.perf_counter()
                try:
                    return fn(*a, **k)
                finally:
                    acc[lab] = acc.get(lab, 0.0) + time.perf_counter() - t0
            setattr(obj, name, w)
            return fn

        targets = [(tr, "train_gen"), (tr, "_stage_host"), (tr, "train_disc_async"), (tr, "train_disc"),
                   (tr.gen_algo, "_iteration"), (tr.logger, "dump"), (tr, "_read_stats")]
        if sync:
            targets += [(sync, "begin_round"), (sync, "end_round")]
        saved = [(o, n, wrap(o, n)) for o, n in targets]
        t0 = time.perf_counter()
        for _ in range(10):
            round_e2e()
        t1 = time.perf_counter()
        th.cuda.synchronize()
        t2 = time.perf_counter()
        for o, n, fn in saved:
            setattr(o, n, fn)
        msg = f"[rank {rank}] e2e 10 rounds: {(t1 - t0) * 100:.3f} ms/round host, +{(t2 - t1) * 1e3:.3f} ms final sync\n"
        for k, v in sorted(acc.items(), key=lambda kv: -kv[1]):
            msg += f"[rank {rank}]   {k:<20s} {v * 100:.3f} ms/round\n"
        sys.stderr.write(msg)
    e2e_ms, e2e_rounds = [], split_rounds(K, 3)
    for k in e2e_rounds:
        if world > 1:
            dist.barrier()
        th.cuda.synchronize()
        ms_e = cuda_time_ms(lambda: [round_e2e() for _ in range(k)])
        if world > 1:
            t = th.tensor([ms_e], device=device)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms_e = float(t)
        e2e_ms.append(ms_e)
    ms_e = statistics.median(m / k for m, k in zip(e2e_ms, e2e_rounds))
    e2e_value = world * E * T / (ms_e / 1e3)

    # ---- roofline: dominant kernel (PPO update) + disc kernel sweep point + stage kernels (rank 0) ------------------------------
    roof, roof_disc, roof_stages, cpu_base = None, None, None, None
    if rank == 0:
        peak, peak_src = peaks()
        gen = tr.gen_algo
        gen.collect_rollouts()
        tr.venv_buffering.discard()
        th.cuda.synchronize()
        reps = 10
        ms_ppo = cuda_time_ms(lambda: [gen.train() for _ in range(reps)]) / reps
        n_rows = E * T
        da_row = 1 if cfg["discrete"] else cfg["d_act"]
        ppo_bytes = cfg["ppo_epochs"] * n_rows * (cfg["d_obs"] + da_row + 3) * 4 + 6 * gen.policy.desc.n_params * 4
        ach = ppo_bytes / (ms_ppo / 1e3) / 1e9
        n_opt = cfg["ppo_epochs"] * ((n_rows + cfg["ppo_minibatch"] - 1) // cfg["ppo_minibatch"])
        roof = {"kernel": f"k_ppo_update (persistent 8-CTA cluster, DSMEM gradient exchange; PPO.train = {n_opt} sequential "
                          "minibatch steps)",
                "bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                # dram__bytes_read.sum + dram__bytes_write.sum of one `ncu --set full` capture of this kernel at the hc
                # configuration (profiles/ncu_ppo_r02c_selected.csv, the kernel as it is at the end of round 2): the rollout
                # table stays in L2
                "traffic": PPO_DRAM_BYTES_NCU if args.config == "hc" else None,
                "peak_source": peak_src, "ms_per_launch": ms_ppo, "share_of_step": ms_ppo / ms_round,
                "algorithmic_bytes_per_launch": ppo_bytes,
                "note": f"latency-bound by construction: {n_opt} dependent optimiser steps of {cfg['ppo_minibatch']} rows each; "
                        "the HBM fraction is reported as required, the figure of merit is us per minibatch step = "
                        f"{ms_ppo * 1e3 / n_opt:.2f}"}
        roof_disc = disc_roofline(tr, peak, device)
        roof_stages = stage_rooflines(tr, cfg, peak)
        if world == 1 and args.cpu_rounds > 0:
            v, spr, cores, table = time_cpu_port(cfg, E, args.cpu_rounds, 1, stages=True)
            cpu_base = {"value": v, "unit": "env-steps/s", "cores": cores, "kind": "port", "stages_ms_per_round": table,
                        "sample": f"{args.cpu_rounds} rounds x {E * T} env steps after 1 warm-up round "
                                  f"({spr * args.cpu_rounds:.1f} s); oracle/gail_port.py, torch threads auto-picked = "
                                  f"{cores} of {os.cpu_count()} host cores (fastest for these tiny tensors)"}

    if rank == 0:
        line = {"metric": "GAIL env-steps/sec (disc+gen loop)" if cfg["algo"] == "gail" else "AIRL env-steps/sec (disc+gen loop)",
                "value": value, "unit": "env-steps/s",
                "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": ms_round,
                "windows_ms": [round(x, 4) for x in win_ms], "windows_steps": win_rounds,
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": config, "clocks": clocks.summary(),
                "e2e": {"value": e2e_value, "unit": "env-steps/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                        "steps": K, "ms_per_step": ms_e, "windows_ms": [round(x, 4) for x in e2e_ms],
                        "windows_steps": e2e_rounds,
                        "path": f"{cfg['algo'].upper()}.train_gen() + .train_disc(expert_samples=<pinned host batch>) -> "
                                "Mapping[str,float]"},
                "gpu_launches": launches, "roofline": roof, "roofline_disc": roof_disc, "roofline_stages": roof_stages,
                "cpu_baseline": cpu_base}
        print(json.dumps(line))
    if world > 1:
        # (collectives captured in CUDA graphs: skip the process-group teardown, which can block on live graph objects)
        sys.stdout.flush()
        sys.stderr.flush()
        th.cuda.synchronize()
        dist.barrier()
        os._exit(0)


if __name__ == "__main__":
    main()
