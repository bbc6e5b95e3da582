"""GPU: the discriminator entry points that share arithmetic agree bit for bit.

Several entry points reach the same RunningNorm update, Adam step and train statistics by different launches: the separate
reduce + Adam kernels and the fused one, one multi-job norm launch and a launch per normaliser (the fallback for batches
whose chunks do not fit one launch), the immediate fold and the deferred slot list.  Each configuration takes one of these
paths, so the equalities are pinned here with torch.equal rather than through tolerances against the reference.
"""
import pytest
import torch as th

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def L():
    from imitation_b200 import _lib

    _lib.lib()
    return _lib


def _batch(Do, Da, n, seed):
    """feature-major disc batch with rows [0, n) filled: features of different means and scales, zero padding"""
    from imitation_b200 import _desc

    bw, ld = _desc.batch_rows(Do, Da), _desc.batch_ld(n)
    g = th.Generator(device="cuda").manual_seed(seed)
    b = th.zeros(bw, ld, device="cuda")
    scale = th.arange(1, bw + 1, device="cuda", dtype=th.float32)[:, None]
    b[:, :n] = th.randn(bw, n, device="cuda", generator=g) * scale + 0.5 * scale
    return b, ld


def _ws_snap_offset(d):
    """float offset of the potential-norm snapshot inside the workspace (mirror of ws_layout in csrc/imb_disc.cu)."""
    return (d.n_params + 31) // 32 * 32 + 64


# ---------------------------------------------------------------------------------------------
# optimiser: disc_reduce + disc_adam == disc_reduce + disc_reduce_adam
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kernel,weight_decay", [("tc", 0.0), ("tc", 1e-2), ("ffma", 0.0), ("ffma", 1e-2),
                                                  ("tc_grad_flat", 0.0)])
def test_separate_and_fused_optimiser_agree(L, kernel, weight_decay):
    """Two updates of two minibatches each; the last minibatch of an update ends either in disc_reduce + disc_adam or in
    the single disc_reduce_adam launch.  Parameters, both moments, the nine statistics and the step counter must be
    identical.  `tc_grad_flat`: the separate path takes the gradient from an external buffer filled by disc_reduce."""
    from imitation_b200 import _desc

    Do, Da, mb = 17, 6, 512
    n = 2 * mb
    d = _desc.disc_desc(Do, Da)
    extra = L.IMB_F_NO_TENSOR if kernel == "ffma" else 0
    batches = [_batch(Do, Da, n, seed) for seed in (1, 2)]
    g = th.Generator(device="cuda").manual_seed(7)
    P0 = (th.rand(d.n_params, device="cuda", generator=g) - 0.5) * 0.6
    opt = L.Adam(lr=1e-3, beta1=0.9, beta2=0.999, eps=1e-8, weight_decay=weight_decay)
    NS = th.zeros(2, device="cuda")

    def run(fused):
        P, M, V = P0.clone(), th.zeros_like(P0), th.zeros_like(P0)
        ws = th.zeros(L.disc_workspace_floats(d), device="cuda")
        st = th.zeros(L.ST_WORDS, dtype=th.int64, device="cuda")
        stats_out = th.zeros(16, device="cuda")
        grad = th.zeros_like(P0) if kernel == "tc_grad_flat" else None
        for _ in range(2):
            for i, (b, ld) in enumerate(batches):
                flags = (L.IMB_F_ZERO_GRAD if i == 0 else 0) | extra
                L.disc_fwd_bwd(d, P, NS, b, ld, n, mb, 1.0 / (2 * n), None, None, flags, ws)
                if fused and i == len(batches) - 1:
                    L.disc_reduce_adam(d, opt, P, M, V, 1.0, ws, st, stats_out)
                else:
                    L.disc_reduce(d, ws, grad)
            if not fused:
                L.disc_adam(d, opt, P, M, V, grad, 1.0, ws, st, stats_out)
        th.cuda.synchronize()
        return P, M, V, stats_out, st[L.ST_DISC_STEP]

    sep, fus = run(False), run(True)
    assert int(sep[4]) == 2
    for name, a, b in zip(("params", "exp_avg", "exp_avg_sq", "stats_out", "step"), sep, fus):
        assert th.equal(a, b), name


# ---------------------------------------------------------------------------------------------
# RunningNorm: one multi-job launch == three single-normaliser launches; immediate == deferred + fold
# ---------------------------------------------------------------------------------------------
def _norm_init(Do, Da):
    """a running state that is not the fresh (0, 1, 0) one, so the fold's every term matters"""
    g = th.Generator(device="cuda").manual_seed(11)
    nf = 2 * (Do + Da) + 2 * Do
    ns = th.rand(nf, device="cuda", generator=g) + 0.25
    nc = th.tensor([5000, 7000], dtype=th.int32, device="cuda")
    return ns, nc


@pytest.mark.parametrize("n", [1000, 16384, 3_000_000])
def test_multi_job_norm_update_matches_sequential(L, n):
    """A shaped net's disc_norm_update (base normaliser; potential's with next_obs, then with obs) equals three
    norm_batch_stats calls in that order, including the snapshot the Phi(s') pass reads.  3 000 000 rows need more chunks
    than one launch holds for three jobs, so that size takes the one-launch-per-job branch."""
    from imitation_b200 import _desc

    Do, Da = 4, 2
    d = _desc.disc_desc(Do, Da, normalize_input=True, shaped=True)
    assert d.base.norm_off == 0 and d.potential.norm_off == 2 * (Do + Da)
    assert d.base.count_idx == 0 and d.potential.count_idx == 1
    b, ld = _batch(Do, Da, n, n)
    ns, nc = _norm_init(Do, Da)
    ns_seq, nc_seq = ns.clone(), nc.clone()

    ws = th.zeros(L.disc_workspace_floats(d), device="cuda")
    L.disc_norm_update(d, b, ld, n, ns, nc, ws)
    so = _ws_snap_offset(d)
    snap = ws[so:so + 2 * Do].clone()

    ws_seq = th.zeros_like(ws)
    pot, pot_c = ns_seq[2 * (Do + Da):], nc_seq[1:2]
    L.norm_batch_stats(d, b, ld, n, 0, Do + Da, ns_seq[:2 * (Do + Da)], nc_seq[0:1], None, 0, ws_seq)
    L.norm_batch_stats(d, b, ld, n, Do + Da, Do, pot, pot_c, None, 0, ws_seq)
    snap_seq = pot.clone()
    L.norm_batch_stats(d, b, ld, n, 0, Do, pot, pot_c, None, 0, ws_seq)
    th.cuda.synchronize()

    assert th.equal(ns, ns_seq)
    assert th.equal(nc, nc_seq) and nc.tolist() == [5000 + n, 7000 + 2 * n]
    assert th.equal(snap, snap_seq)


def _immediate_and_deferred(L, n):
    """one normaliser updated from two batches (obs rows, then next_obs rows) by norm_batch_stats folding immediately, and
    a copy updated through the deferred slot list applied by norm_fold.  The running count starts at n + 1000: both
    products of the variance fold have similar magnitudes and var * cnt is never exact (as it is when cnt is a power of
    two), so a rounding difference between the paths shows."""
    from imitation_b200 import _desc

    Do, Da = 17, 6
    d = _desc.disc_desc(Do, Da, normalize_input=True)
    b, ld = _batch(Do, Da, n, n + 1)
    g = th.Generator(device="cuda").manual_seed(13)
    ns = th.rand(2 * Do, device="cuda", generator=g) + 0.25
    nc = th.tensor([n + 1000], dtype=th.int32, device="cuda")
    ns_def, nc_def = ns.clone(), nc.clone()
    ws = th.zeros(L.disc_workspace_floats(d), device="cuda")
    cap = 4
    defer = th.zeros(4 + cap * (2 * Do + 1), device="cuda")
    for row0 in (0, Do + Da):
        L.norm_batch_stats(d, b, ld, n, row0, Do, ns, nc, None, 0, ws)
        L.norm_batch_stats(d, b, ld, n, row0, Do, ns_def, nc_def, defer, cap, ws)
    L.norm_fold(Do, defer, ns_def, nc_def)
    th.cuda.synchronize()
    assert float(defer[0]) == 0.0
    return Do, (ns, nc), (ns_def, nc_def)


@pytest.mark.parametrize("n", [1000, 16384, 3_000_000])
def test_immediate_and_deferred_norm_update_agree_on_mean_and_count(L, n):
    Do, (ns, nc), (ns_def, nc_def) = _immediate_and_deferred(L, n)
    assert th.equal(ns[:Do], ns_def[:Do])
    assert th.equal(nc, nc_def) and int(nc) == 3 * n + 1000


@pytest.mark.xfail(strict=True, reason="nvcc contracts the variance fold var * cnt + b_var * b_n as "
                   "fma(b_var, b_n, var * cnt) in k_norm_stats and fma(var, cnt, b_var * b_n) in k_norm_fold")
@pytest.mark.parametrize("n", [1000, 16384, 3_000_000])
def test_immediate_norm_update_matches_deferred_fold(L, n):
    Do, (ns, nc), (ns_def, nc_def) = _immediate_and_deferred(L, n)
    assert th.equal(ns, ns_def) and th.equal(nc, nc_def)
