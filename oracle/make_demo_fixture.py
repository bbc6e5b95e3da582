"""TEST INFRASTRUCTURE.  Cut small demonstration fixtures in the reference's legacy `.npz` layout (data/serialize.py:50-65:
concatenated obs / acts / infos / rews split at `indices`, one extra observation per trajectory, `terminal` per trajectory)
out of the reference's own on-disk expert rollouts, so that the ingest tests can run where /root/reference does not exist:

    tests/testdata/expert_models/cartpole_0/rollouts/final.npz  -> tests/golden/demo_cartpole_legacy.npz  (first 4 trajectories)
    tests/testdata/expert_models/pendulum_0/rollouts/final.npz  -> tests/golden/demo_pendulum_legacy.npz  (first 3 trajectories)
    and, with every trajectory cut to its first 8 transitions, -> tests/golden/demo_{cartpole,pendulum}_all.npz

Run in the build container:  python oracle/make_demo_fixture.py
"""
import os

import numpy as np

REF = "/root/reference/tests/testdata/expert_models"
OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")


def cut(src, dst, k):
    z = np.load(src, allow_pickle=True)
    idx = np.asarray(z["indices"])
    n_act = int(idx[k - 1]) if k <= len(idx) else len(z["acts"])
    n_obs = n_act + k
    out = dict(obs=z["obs"][:n_obs], acts=z["acts"][:n_act], infos=z["infos"][:n_act], terminal=z["terminal"][:k],
               indices=idx[:k - 1])
    if "rews" in z.files:
        out["rews"] = z["rews"][:n_act]
    with open(dst, "wb") as f:
        np.savez_compressed(f, **out)
    print("wrote", dst, {a: out[a].shape for a in out})


def shrink(src, dst, steps):
    """Every trajectory of `src`, each cut to its first `steps` transitions (and `steps` + 1 observations), in the same
    layout: a small file that still holds all of the reference's trajectories and their `terminal` flags."""
    z = np.load(src, allow_pickle=True)
    idx = np.asarray(z["indices"])
    bounds = np.r_[0, idx, len(z["acts"])]
    keep = [np.arange(a, min(b, a + steps)) for a, b in zip(bounds[:-1], bounds[1:])]
    keep_obs = [np.arange(a + i, a + i + len(k) + 1) for i, (a, k) in enumerate(zip(bounds[:-1], keep))]
    acts_at, obs_at = np.concatenate(keep), np.concatenate(keep_obs)
    out = dict(obs=z["obs"][obs_at], acts=z["acts"][acts_at], infos=z["infos"][acts_at], terminal=z["terminal"],
               indices=np.cumsum([len(k) for k in keep])[:-1])
    if "rews" in z.files:
        out["rews"] = z["rews"][acts_at]
    with open(dst, "wb") as f:
        np.savez_compressed(f, **out)
    print("wrote", dst, {a: out[a].shape for a in out})


# (source under REF, leading trajectories kept, fixture), (source, transitions kept per trajectory, fixture)
CUTS = [("cartpole_0/rollouts/final.npz", 4, "demo_cartpole_legacy"), ("pendulum_0/rollouts/final.npz", 3, "demo_pendulum_legacy")]
SHRINKS = [("cartpole_0/rollouts/final.npz", 8, "demo_cartpole_all"), ("pendulum_0/rollouts/final.npz", 8, "demo_pendulum_all")]

if __name__ == "__main__":
    for src, k, name in CUTS:
        cut(os.path.join(REF, src), os.path.join(OUT, name + ".npz"), k)
    for src, steps, name in SHRINKS:
        shrink(os.path.join(REF, src), os.path.join(OUT, name + ".npz"), steps)
