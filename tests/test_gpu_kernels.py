"""GPU parity tests: every CUDA kernel of libb200rl.so against the CPU oracle (oracle/*.py) on identical inputs.
Integer / index work (flags, tstep, path counts) and PointEnv arithmetic: bit-exact.  Floating point: tolerances
stated per test (float32 kernels vs float64 oracle)."""
import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from oracle import envs as E            # noqa: E402
from oracle import optim as OPT         # noqa: E402
from oracle import philox as PH         # noqa: E402
from oracle import policy as P          # noqa: E402
from oracle import sampler as S         # noqa: E402


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from rllab_b200 import _lib
    _lib.load()                          # fails loudly if the extension is missing
    return torch.device("cuda:0")


def _ops():
    from rllab_b200 import ops
    return ops


def _L():
    from rllab_b200 import _lib
    return _lib


ENVS = ["point", "cartpole", "pendulum", "cartpole_swingup", "double_pendulum"]
try:
    from oracle import planar as _planar      # noqa: F401
    ENVS += ["swimmer", "hopper"]
except Exception:                             # pragma: no cover
    pass


def _mk(env_name, hidden, seed=0):
    env64 = E.make(env_name)
    dims = P.Dims(env64.O, (hidden, hidden), env64.A)
    theta = P.init_params(dims, np.random.RandomState(seed))
    theta += np.random.RandomState(seed + 1).randn(dims.P) * 0.05     # non-zero biases
    theta[-env64.A:] = -0.5 + 0.1 * np.arange(env64.A)               # log_std
    return env64, dims, theta


def _noise(ops, L, env, N, T, dev, seed=3, it=5):
    eps = torch.empty((T, env.A, N), dtype=torch.float32, device=dev)
    ops.fill_noise(eps, T, 0, env.A, N, 0, L.NOISE_NORMAL, seed, it, 0)
    kind = L.NOISE_UNIFORM if env.noise_kind == "uniform" else L.NOISE_NORMAL
    rr = torch.empty((T + 1, env.K, N), dtype=torch.float32, device=dev)
    ops.fill_noise(rr, T + 1, 0, env.K, N, 0, kind, seed, it, 1)
    return eps, rr


def _gpu_rollout(env_name, hidden, N, T, mpl, dev, inject=True, seed=3, it=5):
    ops, L = _ops(), _L()
    env, dims, theta = _mk(env_name, hidden)
    th32 = torch.tensor(theta, dtype=torch.float32, device=dev)
    b = ops.LaneBatch(env.O, env.A, N, T, dev)
    eps, rr = _noise(ops, L, env, N, T, dev, seed, it)
    if inject:
        ops.rollout(L.ENV_KINDS[env_name], th32, hidden, hidden, 1e-6, b, mpl, eps, rr, seed, it)
    else:
        ops.rollout(L.ENV_KINDS[env_name], th32, hidden, hidden, 1e-6, b, mpl, None, None, seed, it)
    torch.cuda.synchronize()
    return env, dims, th32.cpu().numpy().astype(np.float64), b, eps.cpu().numpy(), rr.cpu().numpy()


# ------------------------------------------------------------------------------------------- noise
def test_philox_stream_matches_oracle(dev):
    ops, L = _ops(), _L()
    rows, K, N = 5, 4, 257
    out = torch.empty((rows, K, N), dtype=torch.float32, device=dev)
    ops.fill_noise(out, rows, 2, K, N, 1000, L.NOISE_UNIFORM, 11, 7, 1)
    raw = PH.raw_block(rows, 2, K, N, 1000, 11, 7, 1)
    assert np.array_equal(out.cpu().numpy(), PH.uniform_from_raw(raw))       # integer stream: bit-exact
    ops.fill_noise(out, rows, 2, K, N, 1000, L.NOISE_NORMAL, 11, 7, 0)
    raw = PH.raw_block(rows, 2, K, N, 1000, 11, 7, 0)
    np.testing.assert_allclose(out.cpu().numpy(), PH.normal_from_raw(raw), rtol=5e-5, atol=2e-5)
    big = torch.empty((64, 2, 4096), dtype=torch.float32, device=dev)
    ops.fill_noise(big, 64, 0, 2, 4096, 0, L.NOISE_NORMAL, 1, 0, 0)
    x = big.cpu().numpy().astype(np.float64)
    assert abs(x.mean()) < 5e-3 and abs(x.std() - 1.0) < 5e-3


def _close_frac(a, b, rtol, atol, frac=0.999):
    """allclose for all but a (1-frac) share of elements (chaotic float32 contact dynamics produce rare outliers)."""
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    ok = np.abs(a - b) <= atol + rtol * np.abs(b)
    assert ok.mean() >= frac, (ok.mean(), np.abs(a - b).max())


# ------------------------------------------------------------------------------------------- env step
@pytest.mark.parametrize("env_name", ENVS)
def test_env_step_matches_oracle(dev, env_name):
    ops, L = _ops(), _L()
    env32 = E.make(env_name, np.float32)
    kind = L.ENV_KINDS[env_name]
    info = L.env_info(kind)
    assert (info["obs_dim"], info["act_dim"], info["state_dim"], info["reset_dim"]) == (env32.O, env32.A, env32.S, env32.K)
    N, steps = 512, 25
    rng = np.random.RandomState(0)
    raw = rng.rand(env32.K, N).astype(np.float32) if env32.noise_kind == "uniform" else \
        rng.randn(env32.K, N).astype(np.float32)
    state = torch.empty((env32.S, N), dtype=torch.float32, device=dev)
    obs = torch.empty((env32.O, N), dtype=torch.float32, device=dev)
    rew = torch.empty((N,), dtype=torch.float32, device=dev)
    done = torch.empty((N,), dtype=torch.uint8, device=dev)
    ops.env_reset(kind, N, state, obs, torch.tensor(raw, device=dev))
    s = env32.reset(raw)
    exact = env_name == "point"
    ptol = 20.0 if env_name in ("swimmer", "hopper") else 1.0     # stiff contact / 50 sub-steps in float32
    tol = dict(rtol=0, atol=0) if exact else dict(rtol=2e-4, atol=2e-5)
    np.testing.assert_allclose(obs.cpu().numpy(), env32.obs(s), **tol)
    for t in range(steps):
        a = (rng.randn(env32.A, N) * 0.7).astype(np.float32)
        ops.env_step(kind, N, state, torch.tensor(a, device=dev), obs, rew, done)
        s, r, d = env32.step(s, env32.scale_action(a))
        if exact:
            assert np.array_equal(obs.cpu().numpy(), env32.obs(s))          # PointEnv: bit-identical
            assert np.array_equal(rew.cpu().numpy(), r)
            assert np.array_equal(done.cpu().numpy().astype(bool), d)
        else:
            # re-sync the oracle to the device state each step so that errors do not compound chaotically
            _close_frac(obs.cpu().numpy(), env32.obs(s), 2e-4 * ptol, 5e-5 * ptol)
            _close_frac(rew.cpu().numpy(), r, 2e-4 * ptol, 5e-4 * ptol)
            dd = done.cpu().numpy().astype(bool)
            assert (dd != d).mean() < 0.01
            s = state.cpu().numpy()


# ------------------------------------------------------------------------------------------- fused rollout
@pytest.mark.parametrize("env_name,hidden", [(e, 32) for e in ENVS] + [(e, 64) for e in ENVS])
def test_rollout_matches_oracle(dev, env_name, hidden):
    N, T, mpl = 256, 40, 17
    env, dims, theta, b, eps, rr = _gpu_rollout(env_name, hidden, N, T, mpl, dev)
    env32 = E.make(env_name, np.float32)
    traj = b.to_numpy()
    ref = S.rollout_lanes(env32, theta, dims, N, T, mpl, eps, rr)
    # integer/index work: identical except where a done threshold is within float noise
    mism = (traj["flags"] != ref["flags"]).any(axis=0)
    assert mism.mean() < 0.02
    ok = ~mism
    assert np.array_equal(traj["tstep"][:, ok], ref["tstep"][:, ok])
    planar = env_name in ("swimmer", "hopper")
    tcmp = 6 if planar else T          # planar chains diverge chaotically in float32: compare the first steps only
    for k, tol in (("obs", 2e-3), ("act", 2e-3), ("mean", 2e-3), ("rew", 5e-3)):
        sl = (slice(None), slice(0, tcmp)) if traj[k].ndim == 3 else (slice(0, tcmp),)
        _close_frac(traj[k][sl][..., ok], ref[k][sl][..., ok], tol, tol, 0.999 if planar else 1.0)
    np.testing.assert_allclose(traj["log_std"], ref["log_std"], rtol=1e-6)
    # one-step policy parity at float32 resolution: mean(obs) against the float64 oracle on the DEVICE's obs
    mu, _ = P.forward(theta, traj["obs"].reshape(env.O, -1).T, dims)
    np.testing.assert_allclose(traj["mean"].reshape(env.A, -1).T, mu, rtol=2e-5, atol=2e-6)


@pytest.mark.parametrize("env_name", ENVS)
def test_rollout_replay_index_work_exact(dev, env_name):
    """Replay the device's own recorded actions through the float32 oracle env: PointEnv obs/rew/flags/tstep must be
    bit-identical; the other envs agree to float32 tolerance with identical flags away from thresholds."""
    N, T, mpl = 128, 60, 23
    env, dims, theta, b, eps, rr = _gpu_rollout(env_name, 32, N, T, mpl, dev)
    env32 = E.make(env_name, np.float32)
    traj = b.to_numpy()
    s = env32.reset(rr[0])
    plen = np.zeros(N, np.int64)
    for t in range(T):
        o = env32.obs(s)
        s2, r, d = env32.step(s, env32.scale_action(traj["act"][:, t]))
        plen1 = plen + 1
        whole = d | (plen1 >= mpl)
        end = whole | (t == T - 1)
        fl = d.astype(np.uint8) * 1 + end.astype(np.uint8) * 2 + (end & ~whole).astype(np.uint8) * 4
        if env_name == "point":
            assert np.array_equal(traj["obs"][:, t], o)
            assert np.array_equal(traj["rew"][t], r)
            assert np.array_equal(traj["flags"][t], fl)
            assert np.array_equal(traj["tstep"][t], plen.astype(np.uint16))
        else:
            pt = 20.0 if env_name in ("swimmer", "hopper") else 1.0
            _close_frac(traj["obs"][:, t], o, 1e-4 * pt, 1e-5 * pt, 0.995)
            _close_frac(traj["rew"][t], r, 1e-4 * pt, 2e-4 * pt, 0.995)
            assert (traj["flags"][t] != fl).mean() < 0.02
        # follow the device's bookkeeping so one threshold flip does not cascade
        end_dev = (traj["flags"][t] & 2) != 0
        fresh = env32.reset(rr[t + 1])
        s = np.where(end_dev[None], fresh, s2).astype(np.float32)
        plen = np.where(end_dev, 0, plen1)
    paths = S.lanes_to_paths(traj)
    assert sum(len(p["rewards"]) for p in paths) == N * T                      # every sample belongs to one path
    assert max(len(p["rewards"]) for p in paths) <= mpl


@pytest.mark.parametrize("env_name", ["point", "cartpole"])
def test_rollout_internal_philox_equals_injected(dev, env_name):
    N, T, mpl = 200, 30, 11
    _, _, _, b1, _, _ = _gpu_rollout(env_name, 32, N, T, mpl, dev, inject=True)
    _, _, _, b2, _, _ = _gpu_rollout(env_name, 32, N, T, mpl, dev, inject=False)
    for k in ("obs", "act", "mean", "rew", "flags"):
        assert torch.equal(getattr(b1, k), getattr(b2, k)), k
    assert torch.equal(b1.tstep.view(torch.int16), b2.tstep.view(torch.int16))


def test_policy_get_actions_matches_rollout_forward(dev):
    ops, L = _ops(), _L()
    env, dims, theta = _mk("cartpole", 32)
    th32 = torch.tensor(theta, dtype=torch.float32, device=dev)
    n = 777
    obs = torch.randn((4, n), device=dev)
    eps = torch.randn((1, n), device=dev)
    act = torch.empty((1, n), device=dev)
    mean = torch.empty((1, n), device=dev)
    ls = torch.empty((1,), device=dev)
    ops.policy_get_actions(th32, 4, 32, 32, 1, 1e-6, obs, n, eps, 0, 0, 0, 0, act, mean, ls)
    mu, lsd = P.forward(th32.cpu().numpy().astype(np.float64), obs.cpu().numpy().T.astype(np.float64), dims)
    np.testing.assert_allclose(mean.cpu().numpy().T, mu, rtol=2e-5, atol=2e-6)
    np.testing.assert_allclose(act.cpu().numpy().T, mu + np.exp(lsd) * eps.cpu().numpy().T, rtol=2e-5, atol=2e-6)
    np.testing.assert_allclose(ls.cpu().numpy(), lsd, rtol=1e-6)


# ------------------------------------------------------------------------------------------- process_samples
def _batch_from_numpy(ops, traj, dev):
    O, T, N = traj["obs"].shape
    A = traj["act"].shape[0]
    b = ops.LaneBatch(O, A, N, T, dev)
    b.obs.copy_(torch.tensor(traj["obs"], dtype=torch.float32))
    b.act.copy_(torch.tensor(traj["act"], dtype=torch.float32))
    b.mean.copy_(torch.tensor(traj["mean"], dtype=torch.float32))
    b.rew.copy_(torch.tensor(traj["rew"], dtype=torch.float32))
    b.flags.copy_(torch.tensor(traj["flags"]))
    b.tstep.copy_(torch.tensor(traj["tstep"].view(np.int16)).view(torch.uint16))
    b.log_std.copy_(torch.tensor(traj["log_std"], dtype=torch.float32))
    return b


def _stats_from_device(b):
    s = b.sums.cpu().numpy()
    m = b.maxs.cpu().numpy()
    n_paths = s[3]
    avg_ret = s[5] / n_paths
    vary = s[8] / s[2] - (s[7] / s[2]) ** 2
    varres = s[12] / s[2] - (s[11] / s[2]) ** 2
    return dict(AverageDiscountedReturn=s[4] / n_paths, AverageReturn=avg_ret, NumTrajs=int(round(n_paths)),
                StdReturn=np.sqrt(max(s[6] / n_paths - avg_ret ** 2, 0.0)), MaxReturn=m[0], MinReturn=-m[1],
                ExplainedVariance=1 - varres / (vary + 1e-8),
                adv_mean=s[0] / s[2], adv_std=np.sqrt(max(s[1] / s[2] - (s[0] / s[2]) ** 2, 0.0)))


def test_process_samples_matches_reference_golden(dev, golden):
    """The committed golden vectors were produced by the reference's own BaseSampler.process_samples."""
    ops = _ops()
    g = golden
    traj = {k[len("ps_in_"):]: v for k, v in g.items() if k.startswith("ps_in_") and k != "ps_in_coeffs_prev"}
    # the kernels hold float32 trajectories: feed the reference numbers rounded to float32 and compare at that level
    for tag, coeffs in (("a", None), ("b", g["ps_in_coeffs_prev"]), ("c", g["ps_in_coeffs_prev"])):
        disc, lam, center, positive = g["ps_%s_cfg" % tag]
        b = _batch_from_numpy(ops, traj, dev)
        w = None if coeffs is None else torch.tensor(coeffs, dtype=torch.float64, device=dev)
        ops.process_samples(b, w, disc, lam)
        np.testing.assert_allclose(b.ret.cpu().numpy(), g["ps_%s_ret" % tag], rtol=2e-6, atol=2e-6)
        st = _stats_from_device(b)
        assert st["NumTrajs"] == int(g["ps_%s_NumTrajs" % tag])                      # integer: exact
        for key in ("AverageDiscountedReturn", "AverageReturn", "StdReturn", "MaxReturn", "MinReturn",
                    "ExplainedVariance"):
            np.testing.assert_allclose(st[key], g["ps_%s_%s" % (tag, key)], rtol=5e-5, atol=5e-6, err_msg=key)
        ops.center_advantages(b, bool(center), bool(positive))
        np.testing.assert_allclose(b.adv.cpu().numpy(), g["ps_%s_adv" % tag], rtol=5e-5, atol=5e-5)
        # baseline fit: normal equations on the device, tiny solve on the host exactly as the reference does
        d1 = 2 * b.O + 5
        gram = torch.empty((d1 * (d1 + 1) // 2,), dtype=torch.float64, device=dev)
        ops.lfb_gram(b, gram)
        G = np.zeros((d1, d1))
        G[np.triu_indices(d1)] = gram.cpu().numpy()
        G = G + G.T - np.diag(np.diag(G))
        fit = S.lfb_fit_normal(G[:-1, :-1], G[:-1, -1])
        ref_fit = g["ps_%s_fit" % tag]
        pred_dev = S.lfb_features_lanes(traj["obs"], traj["tstep"]).reshape(d1 - 1, -1).T @ fit
        pred_ref = S.lfb_features_lanes(traj["obs"], traj["tstep"]).reshape(d1 - 1, -1).T @ ref_fit
        np.testing.assert_allclose(pred_dev, pred_ref, rtol=2e-3, atol=2e-3)   # ill-conditioned d=10 on 161 samples
        # ... and the product's device-side solve (b200rl_lfb_solve) against the reference's fit as well
        w_dev = torch.empty((d1 - 1,), dtype=torch.float64, device=dev)
        info = torch.zeros((3,), dtype=torch.float64, device=dev)
        ops.lfb_solve(b.O, gram, 1e-5, w_dev, info)
        assert info.cpu().tolist() == [1e-5, 0.0, 1.0]
        pred_solve = S.lfb_features_lanes(traj["obs"], traj["tstep"]).reshape(d1 - 1, -1).T @ w_dev.cpu().numpy()
        np.testing.assert_allclose(pred_solve, pred_ref, rtol=2e-3, atol=2e-3)


@pytest.mark.parametrize("drop_cut", [False, True], ids=["keep-cut", "drop-cut"])
@pytest.mark.parametrize("N,T", [(4099, 101), (4096, 128)], ids=["unaligned", "aligned"])
@pytest.mark.parametrize("env_name", ENVS)
def test_process_samples_matches_oracle_large(dev, env_name, N, T, drop_cut):
    """The baseline chain at every compiled obs_dim (2, 3, 4, 6, 13, 20) with a nonzero baseline w: predictor, GAE scan,
    statistics, centring, Gram and the device solve (d = 2O+4 up to 44).  4099 x 101: B % 4 != 0 (scalar predictor,
    unaligned scan); 4096 x 128: the vector predictor and the staged scan.  Both sizes make every Gram kernel's
    grid-stride loop iterate."""
    ops = _ops()
    mpl = 40
    env, dims, theta, b, eps, rr = _gpu_rollout(env_name, 32, N, T, mpl, dev)
    traj = b.to_numpy()
    w = np.random.RandomState(5).randn(2 * env.O + 4) * 0.3
    ops.process_samples(b, torch.tensor(w, dtype=torch.float64, device=dev), 0.99, 0.95, drop_cut_paths=drop_cut)
    ref = S.process_samples_lanes(traj, w, 0.99, 0.95, center_adv=True, drop_cut=drop_cut)
    valid = ref["valid"]
    if drop_cut:
        assert not valid.all()
        assert np.array_equal((b.flags.cpu().numpy() & S.FLAG_MASKED) != 0, ~valid)
    np.testing.assert_allclose(b.ret.cpu().numpy(), ref["ret"], rtol=1e-5, atol=1e-4)
    np.testing.assert_allclose(b.base.cpu().numpy(), ref["base"], rtol=1e-5, atol=1e-4)
    np.testing.assert_allclose(b.adv.cpu().numpy(), ref["adv_raw"], rtol=1e-5, atol=2e-4)
    st = _stats_from_device(b)
    for key in ("AverageDiscountedReturn", "AverageReturn", "StdReturn", "MaxReturn", "MinReturn", "ExplainedVariance",
                "adv_mean", "adv_std"):
        np.testing.assert_allclose(st[key], ref["stats"][key], rtol=1e-6, atol=1e-6, err_msg=key)
    assert st["NumTrajs"] == ref["stats"]["NumTrajs"]
    assert b.sums.cpu().numpy()[2] == valid.sum()
    ops.center_advantages(b, True, False)
    np.testing.assert_allclose(b.adv.cpu().numpy(), ref["adv"], rtol=1e-4, atol=1e-5)
    d1 = 2 * b.O + 5
    gram = torch.empty((d1 * (d1 + 1) // 2,), dtype=torch.float64, device=dev)
    ops.lfb_gram(b, gram)
    keep = valid.reshape(-1)
    F = S.lfb_features_lanes(traj["obs"], traj["tstep"]).reshape(d1 - 1, -1)
    F = np.concatenate([F, ref["ret"].reshape(1, -1)], axis=0)[:, keep]
    G = (F @ F.T)[np.triu_indices(d1)]
    np.testing.assert_allclose(gram.cpu().numpy(), G, rtol=2e-5, atol=1e-3)
    # device solve == the reference's lstsq on the same regularised normal equations
    w_dev = torch.empty((d1 - 1,), dtype=torch.float64, device=dev)
    info = torch.zeros((3,), dtype=torch.float64, device=dev)
    ops.lfb_solve(b.O, gram, 1e-5, w_dev, info)
    reg, _, ok = info.cpu().tolist()
    assert ok == 1.0
    Gf = np.zeros((d1, d1))
    Gf[np.triu_indices(d1)] = gram.cpu().numpy()
    Gf = Gf + Gf.T - np.diag(np.diag(Gf))
    w_ref = S.lfb_fit_normal(Gf[:-1, :-1], Gf[:-1, -1], reg)
    Fm = F[:-1].T
    np.testing.assert_allclose(Fm @ w_dev.cpu().numpy(), Fm @ w_ref, rtol=1e-6, atol=1e-6)


def test_lfb_solve_regularisation_retry(dev):
    """linear_feature_baseline.py:30-37: reg *= 10 while the solve fails; at most 5 attempts."""
    ops = _ops()
    O = 2
    d1 = 2 * O + 5
    rs = np.random.RandomState(3)
    X = rs.randn(d1, 3)
    G = X @ X.T - 2e-4 * np.eye(d1)       # rank 3 minus 2e-4 I: positive definite only once reg >= 1e-3 (3rd attempt)
    gram = torch.tensor(G[np.triu_indices(d1)], dtype=torch.float64, device=dev)
    w = torch.empty((d1 - 1,), dtype=torch.float64, device=dev)
    info = torch.zeros((3,), dtype=torch.float64, device=dev)
    ops.lfb_solve(O, gram, 1e-5, w, info)
    reg, attempts, ok = info.cpu().tolist()
    assert ok == 1.0 and attempts == 2.0 and abs(reg - 1e-3) < 1e-15
    A = G[:-1, :-1] + reg * np.eye(d1 - 1)
    np.testing.assert_allclose(A @ w.cpu().numpy(), G[:-1, -1], rtol=1e-6, atol=1e-6)
    # a NaN Gram matrix exhausts the 5 attempts and reports failure
    gram[3] = float("nan")
    ops.lfb_solve(O, gram, 1e-5, w, info)
    assert info.cpu().tolist()[1:] == [5.0, 0.0]


# ------------------------------------------------------------------------------------------- update kernels
def _update_setup(dev, env_name, hidden, N=512, T=32):
    ops = _ops()
    env, dims, theta, b, eps, rr = _gpu_rollout(env_name, hidden, N, T, 20, dev)
    traj = b.to_numpy()
    ops.process_samples(b, None, 0.99, 1.0)
    ops.center_advantages(b, True, False)
    torch.cuda.synchronize()
    batch = S.batch_from_traj(traj, b.adv.cpu().numpy())
    return ops, env, dims, theta, b, batch


@pytest.mark.parametrize("env_name,hidden", [("cartpole", 32), ("point", 32), ("pendulum", 32), ("double_pendulum", 32), ("cartpole", 64)] +
                         ([("swimmer", 32), ("hopper", 64)] if "hopper" in ENVS else []))
def test_loss_kl_grad_fvp_match_oracle(dev, env_name, hidden):
    _check_update_kernels(dev, env_name, hidden, 512, 32)


@pytest.mark.parametrize("env_name,hidden", [("cartpole", 32), ("cartpole", 64)])
def test_update_kernels_ragged_batch(dev, env_name, hidden):
    """B = 509 * 31 = 15 779 samples: odd (activation-cache rows unaligned -> scalar cache path) and not a multiple of the
    128-sample tile (the last tile is partly masked)."""
    _check_update_kernels(dev, env_name, hidden, 509, 31)


def _check_update_kernels(dev, env_name, hidden, N, T):
    L = _L()
    ops, env, dims, theta, b, batch = _update_setup(dev, env_name, hidden, N, T)
    dd = (env.O, hidden, hidden, env.A)
    B = b.B
    th32 = torch.tensor(theta, dtype=torch.float32, device=dev)
    out = torch.zeros(3, dtype=torch.float64, device=dev)
    # at theta_old: 64-wide nets -- likelihood ratio == 1 exactly (the FFMA loss kernel shares the rollout's summation
    # order); 32-wide nets -- the loss pass runs its forward on the tensor cores (3xTF32): the rollout's mean to ~1e-7
    ops.loss_kl(L.LOSS_TRPO, th32, dd, 1e-6, b, out)
    o = out.cpu().numpy()
    if hidden == 64:
        assert abs(o[0] + batch["adv"].mean()) < 1e-9 and abs(o[1]) < 1e-12 and abs(o[2]) < 1e-12
    else:
        assert abs(o[0] + batch["adv"].mean()) < 1e-6 and abs(o[1]) < 1e-10 and abs(o[2]) < 1e-8
    # perturbed parameters: loss / KL / gradient against the float64 oracle
    rng = np.random.RandomState(9)
    th2 = theta + rng.randn(dims.P) * 0.02
    th2_32 = torch.tensor(th2, dtype=torch.float32, device=dev)
    th2 = th2_32.cpu().numpy().astype(np.float64)
    for kind, name in ((L.LOSS_TRPO, "trpo"), (L.LOSS_VPG, "vpg")):
        ops.loss_kl(kind, th2_32, dd, 1e-6, b, out)
        o = out.cpu().numpy()
        ref_loss = P.surr_loss_trpo(th2, batch, dims) if name == "trpo" else P.surr_loss_vpg(th2, batch, dims)
        mkl, xkl = P.kl_stats(th2, batch, dims)
        np.testing.assert_allclose(o[0], ref_loss, rtol=2e-5, atol=2e-6)
        np.testing.assert_allclose(o[1], mkl, rtol=2e-5, atol=1e-8)
        np.testing.assert_allclose(o[2], xkl, rtol=1e-4, atol=1e-8)
        g = torch.zeros(dims.P, dtype=torch.float64, device=dev)
        out_g = torch.zeros(3, dtype=torch.float64, device=dev)
        ops.grad(kind, th2_32, dd, 1e-6, b, g, out_g)
        og = out_g.cpu().numpy()     # fused loss/KL triple (tensor-core forward for 32-wide nets): same oracle tolerances
        np.testing.assert_allclose(og[0], ref_loss, rtol=2e-5, atol=2e-6)
        np.testing.assert_allclose(og[1], mkl, rtol=2e-5, atol=1e-8)
        np.testing.assert_allclose(og[2], xkl, rtol=1e-4, atol=1e-8)
        np.testing.assert_allclose(og, o, rtol=1e-4, atol=2e-6)
        ref_g = P.grad_surr(th2, batch, dims, name)
        # three-pass TF32 chain (tensor cores): 4e-7 of the scale of the summands, i.e. a few 1e-6 of the largest entry
        np.testing.assert_allclose(g.cpu().numpy(), ref_g, rtol=2e-4, atol=5e-6 * np.abs(ref_g).max() + 1e-9)
    # Fisher-vector product at theta_old
    x = rng.randn(dims.P)
    xd = torch.tensor(x, dtype=torch.float64, device=dev)
    Hx = torch.zeros(dims.P, dtype=torch.float64, device=dev)
    ops.fvp(th32, dd, 1e-6, b, xd, 1e-5, 1.0, Hx)
    # activation cache: the gradient pass at theta_old stores tanh outputs, the FVP reads them back -> identical result
    hc = b.hcache(hidden, hidden)
    gtmp = torch.zeros(dims.P, dtype=torch.float64, device=dev)
    ops.grad(L.LOSS_TRPO, th32, dd, 1e-6, b, gtmp, None, hc)
    Hx_c = torch.zeros(dims.P, dtype=torch.float64, device=dev)
    ops.fvp(th32, dd, 1e-6, b, xd, 1e-5, 1.0, Hx_c, hc)
    # with a cache the dense chain runs on the tensor cores (update_umma32.cu / update_umma.cu: three-pass TF32 split,
    # float32 accumulation in TMEM): float32-grade agreement with the FFMA kernel, not bit equality -- and the same
    # agreement with the float64 oracle as the FFMA kernel
    if True:
        np.testing.assert_allclose(Hx_c.cpu().numpy(), Hx.cpu().numpy(), rtol=0, atol=5e-6 * np.abs(Hx.cpu().numpy()).max())
        ref_c = P.fvp(theta, batch, x.astype(np.float32).astype(np.float64), dims, 0.0) + 1e-5 * x
        np.testing.assert_allclose(Hx_c.cpu().numpy(), ref_c, rtol=2e-4, atol=2e-6 * np.abs(ref_c).max())
    x32 = x.astype(np.float32).astype(np.float64)          # the kernel rounds the tangent to float32
    ref_Hx = P.fvp(theta, batch, x32, dims, 0.0) + 1e-5 * x
    np.testing.assert_allclose(Hx.cpu().numpy(), ref_Hx, rtol=2e-4, atol=2e-6 * np.abs(ref_Hx).max())


def test_min_std_clamp_blocks_logstd_gradient(dev):
    L = _L()
    ops, env, dims, theta, b, batch = _update_setup(dev, "cartpole", 32)
    th = theta.copy()
    th[-1] = np.log(1e-3) - 1.0            # below log(min_std=1e-3)
    dd = (env.O, 32, 32, env.A)
    g = torch.zeros(dims.P, dtype=torch.float64, device=dev)
    th32 = torch.tensor(th, dtype=torch.float32, device=dev)
    ops.grad(L.LOSS_VPG, th32, dd, 1e-3, b, g)
    ref = P.grad_surr(th32.cpu().numpy().astype(np.float64), batch, dims, "vpg", min_std=1e-3)
    assert g.cpu().numpy()[-1] == 0.0 and ref[-1] == 0.0
    np.testing.assert_allclose(g.cpu().numpy(), ref, rtol=5e-4, atol=1e-6 * np.abs(ref).max() + 1e-9)


# ------------------------------------------------------------------------------------------- vector kernels
def test_cg_kernels_match_reference_golden(dev, golden):
    ops = _ops()
    A = torch.tensor(golden["cg_A"], dtype=torch.float64, device=dev)
    bvec = torch.tensor(golden["cg_b"], dtype=torch.float64, device=dev)
    for iters, key in ((10, "cg_x10"), (3, "cg_x3")):
        x, r, p = (torch.empty_like(bvec) for _ in range(3))
        st = torch.zeros(4, dtype=torch.float64, device=dev)
        ops.cg_init(bvec, x, r, p, st)
        for _ in range(iters):
            z = (A @ p).contiguous()      # test plumbing only: the product path uses b200rl_fvp here
            ops.cg_step(z, x, r, p, st)
        np.testing.assert_allclose(x.cpu().numpy(), golden[key], rtol=1e-9, atol=1e-12)
    # early exit emulation: once rdotr < tol the state freezes (krylov.py:36-37 break)
    x, r, p = (torch.empty_like(bvec) for _ in range(3))
    st = torch.zeros(4, dtype=torch.float64, device=dev)
    ops.cg_init(bvec, x, r, p, st)
    for _ in range(40):
        ops.cg_step((A @ p).contiguous(), x, r, p, st, 1e-10)
    ref = OPT.cg(lambda v: golden["cg_A"] @ v, golden["cg_b"].copy(), 40)
    np.testing.assert_allclose(x.cpu().numpy(), ref, rtol=1e-7, atol=1e-10)
    assert st.cpu().numpy()[1] == 1.0 and st.cpu().numpy()[3] < 40


def test_step_size_axpy_adam_match_oracle(dev):
    ops = _ops()
    rng = np.random.RandomState(2)
    Pn = 1250
    x, Hx, th = rng.randn(Pn), rng.randn(Pn), rng.randn(Pn)
    Hx = np.abs(Hx) * np.sign(x)          # x.Hx > 0
    xd, Hd, td = (torch.tensor(v, dtype=torch.float64, device=dev) for v in (x, Hx, th))
    step = torch.empty_like(xd)
    info = torch.zeros(2, dtype=torch.float64, device=dev)
    ops.trpo_step_size(xd, Hd, 0.01, step, info)
    beta = np.sqrt(2.0 * 0.01 * (1.0 / (x.dot(Hx) + 1e-8)))
    np.testing.assert_allclose(info.cpu().numpy()[0], beta, rtol=1e-12)
    np.testing.assert_allclose(step.cpu().numpy(), beta * x, rtol=1e-12)
    ops.trpo_step_size(xd, -Hd, 0.01, step, info)            # negative curvature -> NaN -> 1 (cg_opt.py:264-265)
    assert info.cpu().numpy()[0] == 1.0
    out64 = torch.empty_like(td)
    out32 = torch.empty(Pn, dtype=torch.float32, device=dev)
    ops.axpy_params(td, step, 0.8 ** 3, out64, out32)
    np.testing.assert_allclose(out64.cpu().numpy(), th - 0.8 ** 3 * step.cpu().numpy(), rtol=1e-12)
    assert np.array_equal(out32.cpu().numpy(), out64.cpu().numpy().astype(np.float32))
    m = torch.zeros_like(td)
    v = torch.zeros_like(td)
    th_o, m_o, v_o, t_o = th.copy(), np.zeros(Pn), np.zeros(Pn), 0
    for t in range(1, 4):
        g = rng.randn(Pn)
        ops.adam_step(td, out32, torch.tensor(g, dtype=torch.float64, device=dev), m, v, t)
        th_o, m_o, v_o, t_o = P.adam_step(th_o, g, m_o, v_o, t_o)
    np.testing.assert_allclose(td.cpu().numpy(), th_o, rtol=1e-12)


@pytest.mark.parametrize("env_name,hidden", [("cartpole", 32), ("point", 32), ("cartpole", 64)])
def test_f64_parity_kernels_match_oracle(dev, env_name, hidden):
    """b200rl_update_f64 (float64 arithmetic on the float64 master parameters) vs the float64 oracle: 1e-9."""
    L = _L()
    ops, env, dims, theta, b, batch = _update_setup(dev, env_name, hidden)
    dd = (env.O, hidden, hidden, env.A)
    B = b.B
    rng = np.random.RandomState(4)
    th = theta + rng.randn(dims.P) * 0.02                     # NOT rounded to float32
    thd = torch.tensor(th, dtype=torch.float64, device=dev)
    out = torch.zeros(3, dtype=torch.float64, device=dev)
    g = torch.zeros(dims.P, dtype=torch.float64, device=dev)
    for kind, name in ((L.LOSS_TRPO, "trpo"), (L.LOSS_VPG, "vpg")):
        ops.update_f64(0, kind, thd, dd, 1e-6, b, None, 0.0, 0.0, None, out)
        ref_loss = P.surr_loss_trpo(th, batch, dims) if name == "trpo" else P.surr_loss_vpg(th, batch, dims)
        mkl, xkl = P.kl_stats(th, batch, dims)
        np.testing.assert_allclose(out.cpu().numpy(), [ref_loss, mkl, xkl], rtol=1e-9, atol=1e-13)
        ops.update_f64(1, kind, thd, dd, 1e-6, b, None, 0.0, 0.0, g, out)
        ref_g = P.grad_surr(th, batch, dims, name)
        np.testing.assert_allclose(g.cpu().numpy(), ref_g, rtol=1e-8, atol=1e-12 * np.abs(ref_g).max())
    x = rng.randn(dims.P)
    xd = torch.tensor(x, dtype=torch.float64, device=dev)
    Hx = torch.zeros(dims.P, dtype=torch.float64, device=dev)
    th0 = torch.tensor(theta, dtype=torch.float64, device=dev)
    ops.update_f64(2, L.LOSS_TRPO, th0, dd, 1e-6, b, xd, 1e-5, 1.0, Hx, None)
    ref_Hx = P.fvp(theta, batch, x, dims, 1e-5)
    np.testing.assert_allclose(Hx.cpu().numpy(), ref_Hx, rtol=1e-8, atol=1e-12 * np.abs(ref_Hx).max())


@pytest.mark.parametrize("O,A", [(6, 1), (13, 2), (20, 3), (4, 1), (3, 1), (2, 2)])
def test_lfb_gram_matches_numpy_on_synthetic_batches(dev, O, A):
    """LinearFeatureBaseline normal equations (linear_feature_baseline.py:19-37) on a synthetic batch for every compiled
    obs_dim: the register-tiled kernel (obs_dim 6 / 13 / 20), the register-triangle kernel (<= 4), ragged sizes (B not a
    multiple of the 128-sample tile or of 4), masked samples, observations beyond the +-10 clip; 4099 x 101 and
    4096 x 128 make the grid-stride loops iterate (the float32 register triangle accumulates over the whole loop)."""
    ops, L = _ops(), _L()
    for N, T in ((200, 37), (128, 64), (333, 5), (4099, 101), (4096, 128)):
        rng = np.random.RandomState(O * 100 + N)
        b = ops.LaneBatch(O, A, N, T, dev)
        obs = (rng.randn(O, T, N) * 6.0).astype(np.float32)
        ts = rng.randint(0, 500, size=(T, N)).astype(np.uint16)
        ret = (rng.randn(T, N) * 30.0).astype(np.float32)
        fl = np.where(rng.rand(T, N) < 0.2, L.FLAG_MASKED, 0).astype(np.uint8)
        b.obs.copy_(torch.tensor(obs)), b.ret.copy_(torch.tensor(ret)), b.flags.copy_(torch.tensor(fl))
        b.tstep.copy_(torch.tensor(ts.view(np.int16)).view(torch.uint16))
        b.masked = True
        d1 = 2 * O + 5
        gram = torch.empty((d1 * (d1 + 1) // 2,), dtype=torch.float64, device=dev)
        ops.lfb_gram(b, gram)
        keep = (fl.reshape(-1) & L.FLAG_MASKED) == 0
        o = np.clip(obs.reshape(O, -1).astype(np.float64), -10, 10)
        al = ts.reshape(-1).astype(np.float64) / 100.0
        F = np.concatenate([o, o ** 2, al[None], al[None] ** 2, al[None] ** 3, np.ones((1, al.size)),
                            ret.reshape(1, -1).astype(np.float64)], axis=0)[:, keep]
        G = (F @ F.T)[np.triu_indices(d1)]
        np.testing.assert_allclose(gram.cpu().numpy(), G, rtol=2e-5, atol=2e-5 * np.abs(G).max())
