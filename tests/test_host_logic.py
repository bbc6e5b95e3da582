"""CPU tests of the host-side logic (no GPU, no compute through libimb.so): data types,
hierarchical logger, descriptor builders, env-parameter twin, fixed-horizon check, and the
multi-GPU round synchronisation on a world_size-2 gloo group."""
import os
import sys

import numpy as np
import pytest
import torch as th
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_transitions_validation_and_flatten():
    from imitation_b200.data import types

    obs = np.arange(12, dtype=np.float32).reshape(4, 3)
    t = types.TrajectoryWithRew(obs=obs, acts=np.zeros((3, 2), np.float32), infos=None, terminal=True,
                                rews=np.ones(3, np.float32))
    tr = types.flatten_trajectories_with_rew([t, t])
    assert len(tr) == 6 and tr.dones.tolist() == [False, False, True] * 2
    np.testing.assert_array_equal(tr.next_obs[:3], obs[1:])
    assert not tr.obs.flags.writeable  # read-only like the reference (data/types.py:524-526)
    with pytest.raises(ValueError, match="dones must be boolean"):
        types.Transitions(obs=obs[:3], acts=np.zeros((3, 2)), infos=np.array([{}] * 3), next_obs=obs[1:],
                          dones=np.zeros(3))
    with pytest.raises(ValueError, match="expected one more observations"):
        types.Trajectory(obs=obs, acts=np.zeros((4, 2)), infos=None, terminal=True)
    arrs = types.as_transition_arrays([t])
    assert set(arrs) == {"obs", "acts", "next_obs", "dones"}


def test_hierarchical_logger_accumulate_means():
    from imitation_b200.util import logger

    lg = logger.configure()
    for v in (1.0, 3.0):
        with lg.accumulate_means("disc"):
            lg.record("disc_loss", v)
            lg.dump(0)
    assert lg.name_to_value["mean/disc/disc_loss"] == 2.0
    assert lg.history[0][1] == {"raw/disc/disc_loss": 1.0}
    lg.dump(1)
    assert "mean/disc/disc_loss" in lg.history[-1][1] and not lg.name_to_value
    with pytest.raises(RuntimeError, match="Nested"):
        with lg.accumulate_means("a"):
            with lg.accumulate_means("b"):
                pass


def test_descriptors_and_layouts():
    from imitation_b200 import _desc

    d = _desc.disc_desc(17, 6)
    assert d.base.din == 23 and d.n_params == 23 * 32 + 32 + 32 * 32 + 32 + 32 + 1 == 1857  # SURVEY a9
    d = _desc.disc_desc(17, 6, hid_sizes=(32,), shaped=True, potential_hid_sizes=(32, 32), normalize_input=True)
    assert d.n_params == 801 + 1665 and d.potential.param_off == 801 and d.potential.norm_off == 46
    assert _desc.batch_ld(1) == 128 and _desc.batch_ld(129) == 256
    pd = _desc.policy_desc(17, 6, False, 32)
    assert pd.n_params == 2 * (17 * 32 + 32 + 32 * 32 + 32) + 6 * 32 + 6 + 32 + 1 + 6
    with pytest.raises(NotImplementedError):
        _desc.disc_desc(17, 6, hid_sizes=(32, 32, 32))
    with pytest.raises(NotImplementedError):
        _desc.disc_desc(70, 6)


def test_env_params_twin_matches_oracle_spec():
    from imitation_b200 import _desc
    from oracle import synth_env

    for Do, Da, seed in ((17, 6, 0), (4, 2, 7)):
        spec = synth_env.SynthEnvSpec(Do, Da, seed=seed)
        want = np.concatenate([spec.A.ravel(), spec.Bm.ravel(), spec.c, spec.w])
        np.testing.assert_array_equal(_desc.synth_env_params(Do, Da, seed), want)


def test_state_dict_keys_match_reference_names():
    from imitation_b200 import spaces
    from imitation_b200.rewards import reward_nets
    from imitation_b200.util import networks
    from tests import golden_util as G

    net = reward_nets.BasicShapedRewardNet(spaces.Box(-1, 1, (17,)), spaces.Box(-1, 1, (6,)),
                                           normalize_input_layer=networks.RunningNorm)
    ref_keys = set(G.sub(G.load("disc_airl_hc"), "init"))
    assert set(net.state_dict()) == ref_keys
    net = reward_nets.BasicRewardNet(spaces.Box(-1, 1, (4,)), spaces.Discrete(2), hid_sizes=(64, 64))
    assert set(net.state_dict()) == set(G.sub(G.load("disc_gail_cartpole"), "init"))
    with pytest.raises(NotImplementedError):
        reward_nets.BasicRewardNet(spaces.Box(-1, 1, (4,)), spaces.Discrete(2), dropout_prob=0.5)


def _sync_worker(rank, world, port, out):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    import torch.distributed as dist

    sys.path.insert(0, ROOT)
    from imitation_b200 import distributed

    dist.init_process_group("gloo", rank=rank, world_size=world)
    th.manual_seed(0)
    params = th.arange(6, dtype=th.float32) + 10 * rank
    mean, var, count = th.zeros(3), th.ones(3), th.zeros(1, dtype=th.int32)
    # common start state with data already in it
    start = th.randn(20, 3, generator=th.Generator().manual_seed(1))
    mean.copy_(start.mean(0)), var.copy_(start.var(0, unbiased=False)), count.fill_(20)
    sync = distributed.RoundSync([params], [distributed.NormStat(mean, var, count)])
    sync.begin_round()
    local = th.randn(7 + rank, 3, generator=th.Generator().manual_seed(2 + rank)) * (1 + rank)
    allx = th.cat([start, local])
    mean.copy_(allx.mean(0)), var.copy_(allx.var(0, unbiased=False)), count.fill_(len(allx))
    sync.end_round()
    out[rank] = (params.clone(), mean.clone(), var.clone(), int(count))
    assert distributed.env_slice(4096, rank, world) == (rank * 2048, 2048)
    dist.destroy_process_group()


def test_round_sync_world2_gloo():
    """N>1 path on CPU: parameters averaged, RunningNorm merged exactly (= stats of the union)."""
    world = 2
    mgr = mp.Manager()
    out = mgr.dict()
    port = 29500 + (os.getpid() % 2000)
    mp.spawn(_sync_worker, args=(world, port, out), nprocs=world, join=True)
    start = th.randn(20, 3, generator=th.Generator().manual_seed(1))
    locs = [th.randn(7 + r, 3, generator=th.Generator().manual_seed(2 + r)) * (1 + r) for r in range(world)]
    union = th.cat([start] + locs)
    for r in range(world):
        p, m, v, c = out[r]
        th.testing.assert_close(p, th.arange(6, dtype=th.float32) + 5.0)
        th.testing.assert_close(m, union.mean(0), rtol=1e-5, atol=1e-6)
        th.testing.assert_close(v, union.var(0, unbiased=False), rtol=1e-5, atol=1e-6)
        assert c == len(union)


def test_demo_ingest_npz_round_trip(tmp_path):
    """data/serialize: the legacy .npz layout (indices-split, one extra observation per trajectory) round-trips and
    flattens into the transition arrays the device expert table is built from."""
    from imitation_b200.data import serialize, types

    rng = np.random.default_rng(0)
    trajs = []
    for n, term in ((5, True), (3, False), (7, True)):
        trajs.append(types.TrajectoryWithRew(obs=rng.standard_normal((n + 1, 4)).astype(np.float32),
                                             acts=rng.integers(0, 2, n), infos=None, terminal=term,
                                             rews=rng.standard_normal(n).astype(np.float32)))
    p = tmp_path / "demos" / "final.npz"
    serialize.save(p, trajs)
    raw = np.load(p, allow_pickle=True)
    np.testing.assert_array_equal(raw["indices"], [5, 8])  # the reference's split points (serialize.py:56-60)
    assert raw["obs"].shape == (5 + 3 + 7 + 3, 4)
    back = serialize.load_with_rewards(p)
    assert len(back) == 3
    for a, b in zip(trajs, back):
        np.testing.assert_array_equal(a.obs, b.obs)
        np.testing.assert_array_equal(a.acts, b.acts)
        np.testing.assert_array_equal(a.rews, b.rews)
        assert a.terminal == b.terminal
    flat = types.flatten_trajectories(back)
    assert len(flat) == 15 and flat.dones.sum() == 2 and flat.dones[4] and flat.dones[14] and not flat.dones[7]
    np.testing.assert_array_equal(flat.next_obs[:5], trajs[0].obs[1:])


def _manual_split(raw):
    """the reference's decoding of the legacy layout (data/serialize.py:50-65), spelled out"""
    idx = np.asarray(raw["indices"])
    return (np.split(raw["obs"], idx + np.arange(len(idx)) + 1), np.split(raw["acts"], idx),
            np.split(raw["rews"], idx) if "rews" in raw.files else None)


def _check_fixture(path):
    import warnings

    from imitation_b200.data import serialize, types

    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        trajs = serialize.load_with_rewards(path)
    raw = np.load(path, allow_pickle=True)
    want_obs, want_acts, want_rews = _manual_split(raw)
    assert len(trajs) == len(want_acts) == len(raw["terminal"])
    for t, o, a, r, term in zip(trajs, want_obs, want_acts, want_rews, raw["terminal"]):
        np.testing.assert_array_equal(t.obs, o)
        np.testing.assert_array_equal(t.acts, a)
        np.testing.assert_array_equal(t.rews, r)
        assert len(t.obs) == len(t.acts) + 1 and t.terminal == bool(term)
    # flatten_trajectories (data/rollout.py:563-621): obs[:-1] / obs[1:], dones only at the end of terminal trajectories
    flat = types.flatten_trajectories(trajs)
    np.testing.assert_array_equal(flat.obs, np.concatenate([o[:-1] for o in want_obs]))
    np.testing.assert_array_equal(flat.next_obs, np.concatenate([o[1:] for o in want_obs]))
    np.testing.assert_array_equal(flat.acts, np.concatenate(want_acts))
    dones = np.concatenate([np.r_[np.zeros(len(a) - 1, bool), bool(t)] for a, t in zip(want_acts, raw["terminal"])])
    np.testing.assert_array_equal(flat.dones, dones)
    return trajs


@pytest.mark.parametrize("name", ["demo_cartpole_legacy", "demo_pendulum_legacy"])
def test_demo_ingest_reads_legacy_npz_fixture(name):
    """Fixtures cut from the reference's own expert rollouts (oracle/make_demo_fixture.py) in the legacy layout."""
    import os

    trajs = _check_fixture(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", name + ".npz"))
    assert len(trajs) in (3, 4)


@pytest.mark.parametrize("rel", ["cartpole_0/rollouts/final.npz", "pendulum_0/rollouts/final.npz"])
def test_demo_ingest_reads_reference_rollouts(rel):
    """Every trajectory of the reference's on-disk expert demonstrations (57 CartPole / 56 Pendulum episodes), each cut
    to its first 8 transitions (oracle/make_demo_fixture.py)."""
    import os

    name = {"cartpole_0/rollouts/final.npz": "demo_cartpole_all", "pendulum_0/rollouts/final.npz": "demo_pendulum_all"}[rel]
    trajs = _check_fixture(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", name + ".npz"))
    assert len(trajs) > 50


# ---- preference comparisons: ensemble members over ranks (host logic on CPU, kernels replaced by stand-ins) ------------
def _install_cpu_stand_ins():
    """Replace the CUDA-only pieces by CPU stand-ins whose 'optimiser step' depends on the member's own parameters and on
    exactly which fragment rows, in which order, each minibatch gathered -- so any slip in member assignment, bagging
    subsets, minibatch order (torch RNG bookkeeping for skipped members) or the broadcasts changes the result."""
    from imitation_b200 import _lib
    from imitation_b200.rewards import reward_nets

    E = reward_nets.FusedEngine

    class _Dev:
        type = "cuda"

    def sync(self):
        if getattr(self, "params", None) is not None and getattr(self, "_cpu_synced", False):
            return
        plist = self._param_list()
        flat = th.cat([p.detach().reshape(-1) for p in plist])
        off = 0
        for p in plist:
            p.data = flat[off:off + p.numel()].view(p.shape)
            off += p.numel()
        self.params, self.norm_state, self.norm_count = flat, th.zeros(2), th.zeros(2, dtype=th.int32)
        self.ws = th.zeros(8)
        self._cpu_synced = True

    E.sync = sync
    E.device = lambda self: _Dev()
    E.new_batch = lambda self, n: (th.zeros(4, n), n)
    st = {"h": 0.0}

    def gather_rows(table, cap, tw, idx, n, batch, ld, col0):
        w = th.arange(1, idx.numel() + 1, dtype=th.float64)
        st["h"] = float((idx.double() * w).sum() % 9973) / 9973.0

    def reduce_adam(desc, hp, params, m, v, div, ws, state, out):
        params.mul_(1.0 - hp.lr * hp.weight_decay).add_(1e-3 * st["h"] * (1.0 + params.abs().mean()))
        m.add_(st["h"])
        v.add_(1.0)
        state[_lib.ST_DISC_STEP] += 1

    _lib.gather_rows = gather_rows
    _lib.disc_reduce_adam = reduce_adam
    _lib.disc_adam = lambda desc, hp, params, m, v, g, div, ws, state, out: reduce_adam(desc, hp, params, m, v, div, ws,
                                                                                      state, out)
    for name in ("table_store", "reward_forward", "pref_loss", "disc_fwd_bwd", "disc_reduce", "disc_norm_update"):
        setattr(_lib, name, lambda *a, **k: None)


def _ensemble_run(world_rank=None):
    """Two PreferenceComparisons-style reward-training calls of a 3-member ensemble; returns every member's parameters."""
    from imitation_b200 import spaces
    from imitation_b200.algorithms import preference_comparisons as pc
    from imitation_b200.data import types
    from imitation_b200.rewards import reward_nets

    Do, Da, L, P = 5, 2, 4, 14
    rng = np.random.default_rng(0)
    obs_space, act_space = spaces.Box(-np.inf, np.inf, (Do,)), spaces.Box(-1.0, 1.0, (Da,))

    def frag():
        return types.TrajectoryWithRew(obs=rng.standard_normal((L + 1, Do)).astype(np.float32),
                                       acts=rng.uniform(-1, 1, (L, Da)).astype(np.float32), infos=None, terminal=False,
                                       rews=rng.standard_normal(L).astype(np.float32))

    ds = pc.PreferenceDataset()
    ds.push([(frag(), frag()) for _ in range(P)], (rng.random(P) < 0.5).astype(np.float32))
    th.manual_seed(3)
    members = [reward_nets.BasicRewardNet(obs_space, act_space, hid_sizes=(32, 32)) for _ in range(3)]
    ens = reward_nets.RewardEnsemble(obs_space, act_space, members)
    pm = pc.PreferenceModel(ens)
    pm._pool = pc.FragmentPool(Do, Da, False, "cpu")
    et = pc.EnsembleTrainer(pm, pc.CrossEntropyRewardLoss(), rng=np.random.default_rng(1), batch_size=4, epochs=2, lr=1e-2)
    if world_rank is not None:
        et.set_distributed()
    th.manual_seed(11)
    et.train(ds)
    et.train(ds, epoch_multiplier=1.5)
    probe = float(th.rand(1))  # torch's global RNG must end in the same state on every rank
    return ([m.mlp.dense0.weight.detach().clone() for m in members],
            [float(t.optim.state[m.mlp.dense0.weight]["step"]) for t, m in zip(et.member_trainers, members)],
            [t.optim.state[m.mlp.dense0.weight]["exp_avg"].detach().clone() for t, m in zip(et.member_trainers, members)], probe)


def _ensemble_worker(rank, world, port, out):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    import torch.distributed as dist

    sys.path.insert(0, ROOT)
    _install_cpu_stand_ins()
    dist.init_process_group("gloo", rank=rank, world_size=world)
    out[rank] = _ensemble_run(world_rank=rank)
    dist.destroy_process_group()


def _ensemble_single(_i, out):
    sys.path.insert(0, ROOT)
    _install_cpu_stand_ins()
    out["single"] = _ensemble_run()


def test_member_parallel_ensemble_equals_single_process_world2_gloo():
    """EnsembleTrainer.set_distributed(): member k on rank k % 2, same bagging subsets / minibatch orders as the
    single-process run, owners broadcast parameters + AdamW state: every rank ends bit-identical to the single process."""
    world = 2
    mgr = mp.Manager()
    out = mgr.dict()
    port = 31500 + (os.getpid() % 2000)
    mp.spawn(_ensemble_single, args=(out,), nprocs=1, join=True)
    mp.spawn(_ensemble_worker, args=(world, port, out), nprocs=world, join=True)
    w0, s0, m0, p0 = out["single"]
    assert len({float(w.sum()) for w in w0}) == 3 and all(s > 0 for s in s0)  # the members really trained, differently
    for r in range(world):
        w, s, m, p = out[r]
        assert s == s0 and p == p0, (r, s, s0, p, p0)
        for a, b in zip(w, w0):
            assert th.equal(a, b), f"rank {r}: member parameters differ from the single-process run"
        for a, b in zip(m, m0):
            assert th.equal(a, b), f"rank {r}: AdamW moments differ from the single-process run"


def _fused_bookkeeping(_i, out):
    sys.path.insert(0, ROOT)
    _install_cpu_stand_ins()
    from imitation_b200 import _lib, spaces
    from imitation_b200.algorithms import preference_comparisons as pc
    from imitation_b200.data import types
    from imitation_b200.rewards import reward_nets

    calls = []
    for name in ("gather_rows", "reward_forward", "pref_loss", "disc_fwd_bwd", "disc_reduce", "disc_reduce_adam", "disc_adam"):
        orig = getattr(_lib, name)
        setattr(_lib, name, (lambda nm, f: (lambda *a, **k: (calls.append(nm), f(*a, **k))[1]))(name, orig))
    Do, Da, L, P = 5, 2, 4, 10
    rng = np.random.default_rng(0)
    obs_space, act_space = spaces.Box(-np.inf, np.inf, (Do,)), spaces.Box(-1.0, 1.0, (Da,))

    def frag(n=L):
        return types.TrajectoryWithRew(obs=rng.standard_normal((n + 1, Do)).astype(np.float32),
                                       acts=rng.uniform(-1, 1, (n, Da)).astype(np.float32), infos=None, terminal=False,
                                       rews=rng.standard_normal(n).astype(np.float32))

    ds = pc.PreferenceDataset()
    ds.push([(frag(), frag()) for _ in range(P)], (rng.random(P) < 0.5).astype(np.float32))
    net = reward_nets.BasicRewardNet(obs_space, act_space, hid_sizes=(32, 32))
    pm = pc.PreferenceModel(net, noise_prob=0.05, discount_factor=0.97)
    pm._pool = pc.FragmentPool(Do, Da, False, "cpu")
    tr = pc.BasicRewardTrainer(pm, pc.CrossEntropyRewardLoss(), rng=np.random.default_rng(5), batch_size=6, minibatch_size=3,
                               epochs=3, lr=2e-3)
    res = {"target": tr._fused_target(ds) is not None}
    tr.train(ds)
    res["calls"] = {c: calls.count(c) for c in sorted(set(calls))}
    res["step"] = float(tr.optim.state[net.mlp.dense0.weight]["step"])
    res["aliased"] = (tr.optim.state[net.mlp.dense0.weight]["exp_avg"].data_ptr() == tr._fused_opt["m"].data_ptr())
    res["keys"] = sorted(k for k in tr.logger.name_to_value if k.startswith("mean/reward/epoch-2"))
    # outside the envelope: ragged fragments, another optimiser, the switch -> the autograd path is chosen
    ragged = pc.PreferenceDataset()
    ragged.push([(frag(), frag(L + 1))], np.ones(1, np.float32))
    res["ragged"] = tr._fused_target(ragged) is None
    tr.optim = th.optim.Adam(net.parameters())
    res["other_optimizer"] = tr._fused_target(ds) is None
    tr.optim = th.optim.AdamW(net.parameters())
    tr.use_fused_step = False
    res["switch"] = tr._fused_target(ds) is None
    out["r"] = res


def test_fused_reward_trainer_bookkeeping_with_stand_in_kernels():
    """The device-only reward-training step (algorithms/preference_comparisons.BasicRewardTrainer._train_fused), host side:
    10 pairs, minibatch 3, batch 6, 3 epochs -> per epoch minibatches of 3, 3, 3, 1 pairs = one full-batch optimiser step
    (reduce + AdamW in one launch), then an incomplete batch stepped at the end of the epoch; the torch optimiser's state
    aliases the flat moments and counts the steps; the envelope checks fall back to the autograd path."""
    mgr = mp.Manager()
    out = mgr.dict()
    mp.spawn(_fused_bookkeeping, args=(out,), nprocs=1, join=True)
    r = out["r"]
    assert r["target"] and r["ragged"] and r["other_optimizer"] and r["switch"]
    assert r["calls"] == {"disc_adam": 3, "disc_fwd_bwd": 12, "disc_reduce": 9, "disc_reduce_adam": 3, "gather_rows": 12,
                          "pref_loss": 24, "reward_forward": 12}
    assert r["step"] == 6.0 and r["aliased"]
    assert r["keys"] == ["mean/reward/epoch-2/train/accuracy", "mean/reward/epoch-2/train/gt_reward_loss",
                         "mean/reward/epoch-2/train/loss"]


def test_demo_ingest_huggingface_directory_round_trip(tmp_path):
    """data/serialize + data/huggingface_utils: `save` writes the reference's on-disk format (a HuggingFace datasets
    directory, one row per trajectory: serialize.py:15-24, huggingface_utils.py:91-157), `load` returns a lazy sequence of
    trajectories over it (serialize.py:37-45); Box and Discrete actions, infos, missing infos, rewards / no rewards,
    slicing, and the error paths of the reference."""
    datasets = pytest.importorskip("datasets")
    from imitation_b200.data import huggingface_utils, serialize, types

    rng = np.random.default_rng(0)

    def traj(n, term, discrete, infos, rew=True):
        kw = dict(obs=rng.standard_normal((n + 1, 4)).astype(np.float32),
                  acts=rng.integers(0, 2, n) if discrete else rng.uniform(-1, 1, (n, 3)).astype(np.float32),
                  infos=np.array([{"t": i, "tag": "x"} for i in range(n)]) if infos else None, terminal=term)
        return types.TrajectoryWithRew(rews=rng.standard_normal(n).astype(np.float32), **kw) if rew else types.Trajectory(**kw)

    for discrete in (True, False):
        trajs = [traj(5, True, discrete, True), traj(3, False, discrete, False), traj(7, True, discrete, True)]
        p = tmp_path / f"demos_{int(discrete)}"
        serialize.save(p, trajs)
        assert sorted(os.listdir(p)) == ["data-00000-of-00001.arrow", "dataset_info.json", "state.json"]
        raw = datasets.load_from_disk(str(p))  # the reference's schema: one row per trajectory
        assert set(raw.features) == {"obs", "acts", "infos", "terminal", "rews"} and len(raw) == 3
        assert raw[0]["infos"][2] in ('{"t": 2, "tag": "x"}', '{"tag": "x", "t": 2}') and raw[1]["infos"] == ["{}"] * 3
        back = serialize.load_with_rewards(p)
        assert isinstance(back, huggingface_utils.TrajectoryDatasetSequence) and len(back) == 3
        for a, b in zip(trajs, back):
            assert type(b) is types.TrajectoryWithRew and b.terminal == a.terminal
            np.testing.assert_array_equal(b.obs, a.obs)
            assert b.obs.dtype == np.float32
            np.testing.assert_array_equal(b.acts, a.acts)
            np.testing.assert_array_equal(b.rews, a.rews)
            assert list(b.infos) == (list(a.infos) if a.infos is not None else [{}] * len(a))
        assert [len(t) for t in back[1:]] == [3, 7] and len(back[-1]) == 7
        flat = types.flatten_trajectories(list(back))  # what the device expert table is built from
        assert len(flat) == 15 and flat.dones.sum() == 2 and flat.obs.dtype == np.float32
        np.testing.assert_array_equal(flat.next_obs[:5], trajs[0].obs[1:])
        arrays = types.as_transition_arrays(back)  # what GAIL / AIRL(demonstrations=<loaded sequence>) uploads
        assert set(arrays) == {"obs", "acts", "next_obs", "dones"} and arrays["obs"].shape == (15, 4)
        # saving the loaded sequence again writes the same dataset
        q = tmp_path / f"again_{int(discrete)}"
        serialize.save(q, back)
        np.testing.assert_array_equal(serialize.load(q)[2].obs, trajs[2].obs)
    # without rewards: plain trajectories; load_with_rewards refuses them; mixed sequences cannot be saved
    plain = [traj(4, True, False, False, rew=False), traj(2, False, False, True, rew=False)]
    serialize.save(tmp_path / "plain", plain)
    got = serialize.load(tmp_path / "plain")
    assert type(got[0]) is types.Trajectory and len(got[1]) == 2
    with pytest.raises(ValueError, match="TrajectoryWithRew"):
        serialize.load_with_rewards(tmp_path / "plain")
    with pytest.raises(ValueError, match="rewards but not all"):
        serialize.save(tmp_path / "mixed", [plain[0], traj(2, True, False, False)])
