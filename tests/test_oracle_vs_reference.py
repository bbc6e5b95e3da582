"""This repository's host-side API against the reference's: the reference's own functions were run on the seeded inputs of
oracle/api_cases.py by oracle/make_golden.py, and what they returned is stored in tests/golden/reference_api.npz (the
demonstration directories it wrote in tests/golden/hf_reference_*).  Each test runs this repository's functions on the
same inputs and compares.

The last three tests check the provenance of the fixtures themselves -- they regenerate them from the reference's sources
(imported through oracle/_shim) -- and skip where those sources are not present."""
import json
import os

import numpy as np
import pytest

from oracle import refimport
from oracle.api_cases import (HORIZON_SCRIPTS, PREF_SETTINGS, SAMPLE_UNTIL, SAMPLE_UNTIL_BAD, SCHEDULE_RUNS, error,
                              make_dataset_trajectories, make_hf_trajectories, make_rollout_trajectories, validation_cases)

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
REF = np.load(os.path.join(GOLDEN, "reference_api.npz"))
FACTS = json.loads(str(REF["facts"]))


def test_huggingface_demonstration_format_is_interchangeable_with_the_reference(tmp_path):
    """f3: a demonstration directory written by the REFERENCE's `data.serialize.save` (its `huggingface_utils` over the real
    `datasets` package) is read by `imitation_b200.data.serialize.load`, and this repo's `save` writes the same dataset
    (features and rows) as the reference for the same trajectories -- so the reference's `load` reads it."""
    datasets = pytest.importorskip("datasets")

    from imitation_b200.data import serialize, types

    def same(a, b):
        assert len(a) == len(b)
        for x, y in zip(a, b):
            np.testing.assert_array_equal(np.asarray(x.obs, dtype=np.float32), np.asarray(y.obs, dtype=np.float32))
            np.testing.assert_array_equal(np.asarray(x.acts), np.asarray(y.acts))
            np.testing.assert_array_equal(np.asarray(x.rews, dtype=np.float32), np.asarray(y.rews, dtype=np.float32))
            assert bool(x.terminal) == bool(y.terminal)
            xi = [{}] * len(x.acts) if x.infos is None else list(x.infos)
            yi = [{}] * len(y.acts) if y.infos is None else list(y.infos)
            assert xi == yi

    rng = np.random.default_rng(3)
    for discrete in (False, True):
        trajs = make_hf_trajectories(types, rng, discrete)
        theirs = os.path.join(GOLDEN, f"hf_reference_{int(discrete)}")
        same(trajs, serialize.load_with_rewards(theirs))                   # the reference wrote, this repo reads
        serialize.save(tmp_path / f"ours_{int(discrete)}", trajs)          # this repo writes what the reference wrote
        ours, want = datasets.load_from_disk(str(tmp_path / f"ours_{int(discrete)}")), datasets.load_from_disk(theirs)
        assert ours.features == want.features
        assert ours.to_dict() == want.to_dict()
        same(trajs, serialize.load_with_rewards(tmp_path / f"ours_{int(discrete)}"))


def test_host_side_rollout_helpers_agree_with_the_reference():
    """f4: `rollout_stats` (with and without Monitor infos), `discounted_sum`, the sample-until predicates and
    `flatten_trajectories_with_rew` of imitation_b200.data.rollout against the reference's own functions
    (data/rollout.py:193-286, 509-621, 728-745) on the same random trajectories."""
    from imitation_b200.data import rollout, types

    rng = np.random.default_rng(5)
    for monitor in (False, True):
        ours = make_rollout_trajectories(types, rng, monitor)
        want, got = FACTS[f"rollout_stats/{int(monitor)}"], rollout.rollout_stats(ours)
        assert set(got) == set(want) and ("monitor_return_mean" in want) == monitor
        for k in want:
            assert got[k] == want[k] and type(got[k]) is type(want[k]), k
        fg = rollout.flatten_trajectories_with_rew(ours)
        for field in ("obs", "acts", "next_obs", "dones", "rews"):
            np.testing.assert_array_equal(getattr(fg, field), REF[f"flatten/{int(monitor)}/{field}"], err_msg=field)
        assert [rollout.make_sample_until(**kw)(ours) for kw in SAMPLE_UNTIL] == FACTS[f"sample_until/{int(monitor)}"]
    assert [error(lambda: rollout.make_sample_until(**kw)) for kw in SAMPLE_UNTIL_BAD] == FACTS["sample_until_errors"]
    arr = rng.standard_normal((7, 3))
    np.testing.assert_array_equal(arr, REF["discounted_sum/input"])
    for gamma in (1.0, 0.9):
        np.testing.assert_allclose(rollout.discounted_sum(arr, gamma), REF[f"discounted_sum/{gamma}/2d"], rtol=1e-12)
        np.testing.assert_allclose(rollout.discounted_sum(arr[:, 0], gamma), REF[f"discounted_sum/{gamma}/1d"], rtol=1e-12)


def test_fixed_horizon_check_agrees_with_the_reference():
    """a21: BaseImitationAlgorithm._check_fixed_horizon (algorithms/base.py:69-108): same accept / reject decisions, same
    remembered horizon and the same error text as the reference's class over sequences of episode lengths."""
    from imitation_b200.algorithms import base

    class Ours(base.BaseImitationAlgorithm):
        pass

    for allow in (False, True):
        for script, want in zip(HORIZON_SCRIPTS, FACTS[f"fixed_horizon/{int(allow)}"]):
            algo, events = Ours(allow_variable_horizon=allow), []
            for horizons in script:
                try:
                    algo._check_fixed_horizon(horizons)
                except ValueError as e:
                    events.append(["err", str(e)])
                    break
                events.append(["ok", algo._horizon])
            assert events == want, (allow, script)


def test_trajectory_and_transition_validation_agrees_with_the_reference():
    """data/types.py:61-330: the same inputs are rejected with the same messages by this repo's Trajectory / TrajectoryWithRew /
    Transitions and by the reference's."""
    from imitation_b200.data import types as M

    cases, ok = validation_cases()
    for name, (cls, kw) in cases.items():
        assert error(lambda: getattr(M, cls)(**kw)) == FACTS["validation"][name], name
    assert len(M.Transitions(**ok)) == FACTS["transitions_len"] == 3


def test_comparison_schedule_helpers_agree_with_the_reference():
    """f1: the per-iteration comparison counts of PreferenceComparisons.train (preference_comparisons.py:1622-1636) --
    `util.oric` rounding of the query-schedule shares -- and the named query schedules (:1465-1479)."""
    from imitation_b200.algorithms import preference_comparisons as pc

    rng = np.random.default_rng(0)
    for want in FACTS["oric"]:
        n, total = int(rng.integers(1, 12)), int(rng.integers(0, 300))
        v = rng.random(n) + 1e-3
        x = v / v.sum() * total
        np.testing.assert_array_equal(pc._round_keep_sum(x), np.array(want, dtype=np.int64))
    # seeds handed to samplers / DataLoaders come from the caller's generator the same way
    assert [pc.make_seeds(np.random.default_rng(9), n) for n in (None, 1, 5)] == FACTS["make_seeds"]
    assert set(pc.QUERY_SCHEDULES) == set(FACTS["query_schedules"])
    for name, fn in pc.QUERY_SCHEDULES.items():
        assert [fn(t) for t in np.linspace(0, 1, 7)] == FACTS["query_schedules"][name], name
    # the whole schedule of a run: initial comparisons + oric(shares), as PreferenceComparisons.train computes it
    for name in pc.QUERY_SCHEDULES:
        for total, iters, frac in SCHEDULE_RUNS:
            initial = int(total * frac)
            vec = np.array([pc.QUERY_SCHEDULES[name](t) for t in np.linspace(0, 1, iters)])
            ours = [initial] + [int(v) for v in pc._round_keep_sum(vec / vec.sum() * (total - initial))]
            assert ours == FACTS["schedule_runs"][f"{name}/{total}/{iters}/{frac}"] and sum(ours) == total


def test_reward_net_preprocess_and_registry_agree_with_the_reference():
    """a8 / f4: `RewardNet.preprocess` (reward_nets.py:74-118: float conversion, one-hot Discrete actions) on CPU tensors and
    the registered reward-loader names of rewards/serialize.py:230-260 against the reference's."""
    import torch as th

    from imitation_b200 import spaces
    from imitation_b200.rewards import reward_nets, serialize

    assert sorted(serialize.reward_registry.keys()) == FACTS["reward_registry"]
    rng = np.random.default_rng(0)
    for discrete in (True, False):
        ours = reward_nets.BasicRewardNet(spaces.Box(-1, 1, (4,)), spaces.Discrete(3) if discrete else spaces.Box(-1, 1, (2,)))
        obs, nobs = rng.standard_normal((6, 4)), rng.standard_normal((6, 4)).astype(np.float32)
        acts = rng.integers(0, 3, 6) if discrete else rng.uniform(-1, 1, (6, 2))
        done = rng.random(6) < 0.5
        got = ours.preprocess(obs, acts, nobs, done)
        assert [str(a.dtype) for a in got] == FACTS[f"preprocess/{int(discrete)}/dtypes"]
        for i, a in enumerate(got):
            assert th.equal(a, th.as_tensor(REF[f"preprocess/{int(discrete)}/{i}"]))
        assert {k: list(v.shape) for k, v in ours.state_dict().items()} == FACTS[f"state_dict_shapes/{int(discrete)}"]


def test_trajectory_dataset_and_preference_dataset_agree_with_the_reference(tmp_path):
    """f1 host side: `TrajectoryDataset.sample` (preference_comparisons.py:99-124: shuffled selection with the caller's
    generator), `PreferenceDataset` FIFO / pickling (:909-997) against the reference's classes for the same seeds."""
    from imitation_b200.algorithms import preference_comparisons as pc
    from imitation_b200.data import types

    ours = make_dataset_trajectories(types)
    b = pc.TrajectoryDataset(ours, np.random.default_rng(7))
    for steps in (10, 25, 46, 1):
        tb = b.sample(steps)
        assert [len(t) for t in tb] == FACTS[f"trajectory_sample/{steps}/lens"]
        np.testing.assert_array_equal(np.concatenate([t.obs for t in tb]), REF[f"trajectory_sample/{steps}/obs"])
    assert error(lambda: b.sample(100), RuntimeError) == FACTS["trajectory_sample_error"]
    db, f = pc.PreferenceDataset(max_size=3), ours
    db.push([(f[0], f[1]), (f[2], f[3])], np.array([1.0, 0.0], np.float32))
    db.push([(f[4], f[5]), (f[6], f[0])], np.array([0.5, 1.0], np.float32))
    assert len(db) == FACTS["preference_dataset_len"] == 3
    np.testing.assert_array_equal(db.preferences, REF["preference_dataset/preferences"])
    for i in range(3):
        (xb, yb), pb = db[i]
        assert pb == REF[f"preference_dataset/{i}/pref"]
        assert np.array_equal(xb.obs, REF[f"preference_dataset/{i}/x_obs"])
        assert np.array_equal(yb.acts, REF[f"preference_dataset/{i}/y_acts"])
    db.save(tmp_path / "prefs.pkl")
    back = pc.PreferenceDataset.load(tmp_path / "prefs.pkl")
    assert len(back) == 3 and np.array_equal(back.preferences, db.preferences) and back.max_size == 3
    msgs = [error(lambda: db.push([(f[0], f[1]), (f[2], f[3])], bad))
            for bad in (np.array([1.0], np.float32), np.array([1.0, 0.0], np.float64))]
    assert msgs == FACTS["preference_dataset_errors"]


def test_running_norm_module_and_mode_helpers_agree_with_the_reference():
    """a10: the torch-level `RunningNorm` module (util/networks.py:19-134; the API path and the policy's
    NormalizeFeaturesExtractor use it on whatever device the tensors are on) is bit-identical to the reference's over a
    sequence of training batches and in eval mode; `training()` / `evaluating()` context managers restore the mode."""
    import torch as th

    from imitation_b200.util import networks

    def state_is(m, prefix):
        for k, v in m.state_dict().items():
            assert th.equal(v, th.as_tensor(REF[f"{prefix}/{k}"])), (prefix, k)

    b = networks.RunningNorm(5)
    g = th.Generator().manual_seed(0)
    for step in range(5):
        x = th.randn(7 + step, 5, generator=g) * (1 + step) + step
        assert th.equal(b(x), th.as_tensor(REF[f"running_norm/{step}/y"]))
        state_is(b, f"running_norm/{step}/state")
    b.eval()
    x = th.randn(3, 5, generator=g)
    assert th.equal(b(x), th.as_tensor(REF["running_norm/eval/y"])) and int(b.count) == 45
    state_is(b, "running_norm/eval/state")
    assert {k: str(v.dtype) for k, v in b.state_dict().items()} == FACTS["running_norm_dtypes"]
    prefix = "running_norm/eval/state/"
    b.load_state_dict({k[len(prefix):]: th.as_tensor(REF[k]) for k in REF.files if k.startswith(prefix)})
    for ctx, want in ((networks.training, True), (networks.evaluating, False)):
        b.eval()
        with ctx(b):
            assert b.training is want
        assert b.training is False
        b.train()
        with ctx(b):
            assert b.training is want
        assert b.training is True


def test_preference_probability_and_loss_agree_with_the_reference():
    """f1: `PreferenceModel.probability` (preference_comparisons.py:487-530: discounting, clipping at the threshold, noise
    floor) and the cross-entropy / accuracy arithmetic of `CrossEntropyRewardLoss` (:1043-1090) on CPU tensors against the
    reference's classes, for several (noise_prob, discount_factor, threshold) settings incl. clipped return differences."""
    import torch as th

    from imitation_b200 import spaces
    from imitation_b200.algorithms import preference_comparisons as pc
    from imitation_b200.rewards import reward_nets

    ours_net = reward_nets.BasicRewardNet(spaces.Box(-1, 1, (4,)), spaces.Box(-1, 1, (2,)))
    g = th.Generator().manual_seed(0)
    for i, (noise, discount, threshold) in enumerate(PREF_SETTINGS):
        b = pc.PreferenceModel(ours_net, noise_prob=noise, discount_factor=discount, threshold=threshold)
        for scale in (0.3, 3.0):
            r1, r2 = th.randn(12, generator=g) * scale, th.randn(12, generator=g) * scale
            pb = b.probability(r1, r2)
            assert pb.shape == () and th.equal(pb, th.as_tensor(REF[f"probability/{i}/{scale}"]))
        # a batch of pairs the way the fused path lays it out: [P, L] rewards, time on axis 1
        R1, R2 = th.randn(9, 12, generator=g) * 2, th.randn(9, 12, generator=g) * 2
        batch = b._probability(R1, R2, time_axis=1)
        single = th.as_tensor(REF[f"probability/{i}/pairs"])
        th.testing.assert_close(batch, single, rtol=1e-6, atol=1e-7)
        prefs = (th.rand(9, generator=g) < 0.5).float()
        want = th.as_tensor(REF[f"probability/{i}/bce"])
        th.testing.assert_close(th.nn.functional.binary_cross_entropy(batch, prefs), want, rtol=1e-6, atol=1e-7)
        assert ((batch > 0.5) == (prefs > 0.5)).float().mean() == th.as_tensor(REF[f"probability/{i}/accuracy"])


# ---- provenance of the fixtures: regenerated from the reference's sources ---------------------------------------------
@pytest.mark.refsrc
@pytest.mark.skipif(not refimport.available(), reason="reference sources not present")
def test_goldens_reproduce_from_reference(tmp_path):
    """EVERY file under tests/golden/ is regenerated from the reference's own modules and compared with the committed
    fixture (no golden is taken on trust)."""
    from oracle import make_golden as mg

    mg.OUT = str(tmp_path)
    cases = mg.all_cases()
    committed = sorted(f[:-4] for f in os.listdir(GOLDEN) if f.endswith(".npz") and not f.startswith("demo_"))
    assert sorted(n for n, _ in cases) == committed, "a golden file without a generator (or the reverse)"
    for name, thunk in cases:
        thunk()
        new = np.load(os.path.join(str(tmp_path), name + ".npz"), allow_pickle=True)
        old = np.load(os.path.join(GOLDEN, name + ".npz"), allow_pickle=True)
        assert set(new.files) == set(old.files), name
        for k in old.files:
            if old[k].dtype.kind in "fc":
                np.testing.assert_allclose(new[k], old[k], rtol=1e-6, atol=1e-7, err_msg=f"{name}:{k}")
            elif old[k].dtype.kind == "O":
                assert [str(x) for x in np.ravel(new[k])] == [str(x) for x in np.ravel(old[k])], f"{name}:{k}"
            else:
                np.testing.assert_array_equal(new[k], old[k], err_msg=f"{name}:{k}")
    datasets = pytest.importorskip("datasets")
    for d in (0, 1):
        new = datasets.load_from_disk(os.path.join(str(tmp_path), f"hf_reference_{d}"))
        old = datasets.load_from_disk(os.path.join(GOLDEN, f"hf_reference_{d}"))
        assert new.features == old.features and new.to_dict() == old.to_dict()


@pytest.mark.refsrc
@pytest.mark.skipif(not refimport.available(), reason="reference sources not present")
def test_demo_fixtures_are_cut_from_the_reference_rollouts(tmp_path):
    """tests/golden/demo_*.npz = leading trajectories, or every trajectory shortened, of the reference's own expert
    rollouts (oracle/make_demo_fixture.py)."""
    from oracle import make_demo_fixture as mdf

    made = [(mdf.cut, src, k, name) for src, k, name in mdf.CUTS] + [(mdf.shrink, src, n, name) for src, n, name in mdf.SHRINKS]
    for fn, src, k, name in made:
        out = os.path.join(str(tmp_path), name + ".npz")
        fn(os.path.join(mdf.REF, src), out, k)
        new, old = np.load(out, allow_pickle=True), np.load(os.path.join(GOLDEN, name + ".npz"), allow_pickle=True)
        assert set(new.files) == set(old.files)
        for key in old.files:
            if old[key].dtype.kind == "O":
                assert [str(x) for x in new[key]] == [str(x) for x in old[key]]
            else:
                np.testing.assert_array_equal(new[key], old[key], err_msg=f"{name}:{key}")


@pytest.mark.refsrc
@pytest.mark.skipif(not refimport.available(), reason="reference sources not present")
def test_reference_modules_used_are_the_real_ones():
    im = refimport.load()
    assert im.__file__.startswith(os.path.join(refimport.REF_SRC, "imitation"))
    from imitation.algorithms.adversarial import common

    assert common.__file__ == os.path.join(refimport.REF_SRC, "imitation", "algorithms", "adversarial", "common.py")
