"""Seeded inputs of the reference-API comparisons, shared by oracle/make_golden.py (which runs the reference's own
functions on them and stores the results in tests/golden/reference_api.npz) and tests/test_oracle_vs_reference.py
(which runs this repository's functions on the same inputs).  `T` is the module holding the trajectory types: the
reference's `imitation.data.types` or `imitation_b200.data.types`."""
import numpy as np


def error(fn, exc=ValueError):
    try:
        fn()
    except exc as e:
        return str(e)
    raise AssertionError("no error raised")


def make_hf_trajectories(T, rng, discrete):
    """Trajectories of the demonstration-format test (three lengths, with and without infos)."""
    spec = [(6, True, [{"step": i} for i in range(6)]), (2, False, None), (4, True, [{} for _ in range(4)])]
    return [T.TrajectoryWithRew(obs=rng.standard_normal((n + 1, 5)).astype(np.float32),
                                acts=rng.integers(0, 3, n) if discrete else rng.uniform(-1, 1, (n, 2)).astype(np.float32),
                                infos=None if infos is None else np.array(infos), terminal=term,
                                rews=rng.standard_normal(n).astype(np.float32)) for n, term, infos in spec]


def make_rollout_trajectories(T, rng, monitor):
    """Trajectories of the rollout-helper test; with `monitor`, all but one carry Monitor episode infos."""
    out = []
    for k, n in enumerate(ROLLOUT_LENS):
        rews = rng.standard_normal(n).astype(np.float32)
        infos = None
        if monitor and k != 2:  # one trajectory without infos: it is skipped by the Monitor statistics
            infos = np.array([{} for _ in range(n - 1)] + [{"episode": {"r": float(rews.sum()) + 0.5 * k, "l": n}}])
        out.append(T.TrajectoryWithRew(obs=rng.standard_normal((n + 1, 3)).astype(np.float32), acts=rng.integers(0, 2, n),
                                       infos=infos, terminal=bool(k % 2), rews=rews))
    return out


def make_dataset_trajectories(T):
    r = np.random.default_rng(1)
    return [T.TrajectoryWithRew(obs=r.standard_normal((n + 1, 3)).astype(np.float32), acts=r.integers(0, 2, n), infos=None,
                                terminal=True, rews=r.standard_normal(n).astype(np.float32)) for n in (5, 9, 3, 7, 7, 4, 11)]


def validation_cases():
    """name -> (class name, keyword arguments) that data/types.py rejects."""
    z = np.zeros
    ok = dict(obs=z((3, 2)), acts=z(3), infos=np.array([{}] * 3), next_obs=z((3, 2)), dones=z(3, bool))
    cases = {"traj/len": ("Trajectory", dict(obs=z((3, 2)), acts=z(3), infos=None, terminal=True)),
             "traj/infos": ("Trajectory", dict(obs=z((4, 2)), acts=z(3), infos=np.array([{}] * 2), terminal=True)),
             "traj/empty": ("Trajectory", dict(obs=z((1, 2)), acts=z(0), infos=None, terminal=True))}
    for name, r in {"shape": z((3, 1), np.float32), "dtype": z(3, np.int64)}.items():
        cases["rews/" + name] = ("TrajectoryWithRew", dict(obs=z((4, 2)), acts=z(3), infos=None, terminal=True, rews=r))
    for name, kw in {"next_obs": {**ok, "next_obs": z((3, 3))}, "dones_dtype": {**ok, "dones": z(3)},
                     "dones_shape": {**ok, "dones": z((3, 1), bool)}, "acts": {**ok, "acts": z(2)},
                     "infos": {**ok, "infos": np.array([{}] * 2)}}.items():
        cases["trans/" + name] = ("Transitions", kw)
    return cases, ok


ROLLOUT_LENS = [4, 9, 1, 6, 6]
SAMPLE_UNTIL = [dict(min_timesteps=20), dict(min_episodes=5), dict(min_timesteps=27, min_episodes=2), dict(min_episodes=6)]
SAMPLE_UNTIL_BAD = [dict(), dict(min_timesteps=0), dict(min_episodes=-1)]
HORIZON_SCRIPTS = [[[5, 5], [5], [], [6]], [[3], [3, 3, 4]], [[], [7], [7, 7], [7]], [[2, 9]]]
SCHEDULE_RUNS = ((500, 5, 0.1), (77, 3, 0.25), (1000, 12, 0.1))
PREF_SETTINGS = ((0.0, 1.0, 50.0), (0.1, 0.95, 50.0), (0.3, 0.9, 2.0))
