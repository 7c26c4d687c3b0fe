"""GPU, BASELINE.json full size (cfg2: CartPole, 65 536 lanes x 200 steps = 13.1 M samples): size-independent
properties that need no oracle run -- recurrences, conservation, exactness at theta_old, linearity / symmetry of the
Fisher-vector product, directional-derivative check of the gradient, determinism and sharding invariance of the
counter-based rollout.  torch is used only to check device buffers in place."""
import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

N, T, MPL, H = 65536, 200, 200, 32


@pytest.fixture(scope="module")
def full():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from rllab_b200 import _lib as L, ops
    from oracle import policy as P
    dev = torch.device("cuda:0")
    dims = P.Dims(4, (H, H), 1)
    theta = P.init_params(dims, np.random.RandomState(11))
    theta[-1] = -0.3
    th32 = torch.tensor(theta, dtype=torch.float32, device=dev)
    b = ops.LaneBatch(4, 1, N, T, dev)
    ops.rollout(L.ENV_CARTPOLE, th32, H, H, 1e-6, b, MPL, None, None, 5, 9, 0)
    w = torch.tensor(np.random.RandomState(1).randn(12) * 0.05, dtype=torch.float64, device=dev)
    ops.process_samples(b, w, 0.99, 0.97)
    torch.cuda.synchronize()
    return dict(L=L, ops=ops, dev=dev, dims=dims, th32=th32, b=b, w=w)


def test_rollout_bookkeeping_invariants(full):
    b = full["b"]
    flags = b.flags.to(torch.int32)
    end = (flags & 2) != 0
    done = (flags & 1) != 0
    ts = b.tstep.view(torch.int16).to(torch.int32)
    assert bool(end[-1].all())                                   # the buffer end closes every lane's last path
    assert bool((done <= end).all())                             # done implies end
    assert bool((ts[0] == 0).all())
    nxt = torch.where(end[:-1], torch.zeros_like(ts[1:]), ts[:-1] + 1)
    assert bool((ts[1:] == nxt).all())                           # tstep restarts after every path end, else +1
    assert int((ts == 0).sum()) == int(end.sum())                # one start per end: every sample in exactly one path
    assert int(ts.max()) < MPL
    for k in ("obs", "act", "mean", "rew"):
        assert bool(torch.isfinite(getattr(b, k)).all()), k
    # CartPole: a non-terminal step pays ~10, a terminal one 0 (cartpole_env.py:46-51)
    assert bool((b.rew[done] == 0).all()) and bool((b.rew[~done] > 9.0).all())


def test_returns_and_advantages_satisfy_their_recurrences(full):
    b, w = full["b"], full["w"]
    end = ((b.flags.to(torch.int32) & 2) != 0)
    ret, rew, adv, base = (t.double() for t in (b.ret, b.rew, b.adv, b.base))
    nxt = torch.zeros_like(ret)
    nxt[:-1] = torch.where(end[:-1], torch.zeros_like(ret[1:]), ret[1:])
    assert float((ret - (rew + 0.99 * nxt)).abs().max()) < 2e-3            # float32 storage of values up to ~1e3
    bn = torch.zeros_like(base)
    bn[:-1] = torch.where(end[:-1], torch.zeros_like(base[1:]), base[1:])
    an = torch.zeros_like(adv)
    an[:-1] = torch.where(end[:-1], torch.zeros_like(adv[1:]), adv[1:])
    delta = rew + 0.99 * bn - base
    assert float((adv - (delta + 0.99 * 0.97 * an)).abs().max()) < 2e-3
    s = b.sums.cpu().numpy()
    assert s[2] == N * T and s[3] == float(((b.tstep.view(torch.int16) == 0)).sum())
    np.testing.assert_allclose(s[0], float(adv.sum()), rtol=1e-6)
    full["ops"].center_advantages(b, True, False)
    a = b.adv.double()
    assert abs(float(a.mean())) < 1e-6 and abs(float(a.std(unbiased=False)) - 1.0) < 1e-5


def test_loss_and_kl_at_theta_old(full):
    """At theta_old the surrogate is -mean(adv) and the KL is 0.  The 32-wide update passes run their forward on the
    tensor cores (3xTF32 split, update_umma32.cu), so this holds to float32 rounding of the mean (1e-7), not bit for bit as
    with the FFMA kernels of round 1; the loss pass and the gradient pass share one forward and agree with each other
    far below that."""
    L, ops, b, th32 = full["L"], full["ops"], full["b"], full["th32"]
    out = torch.zeros(3, dtype=torch.float64, device=full["dev"])
    ops.loss_kl(L.LOSS_TRPO, th32, (4, H, H, 1), 1e-6, b, out)
    o = out.cpu().numpy()
    assert abs(o[0] + float(b.adv.double().mean())) < 1e-6 and abs(o[1]) < 1e-10 and abs(o[2]) < 1e-8
    g = torch.zeros(full["dims"].P, dtype=torch.float64, device=full["dev"])
    out2 = torch.zeros(3, dtype=torch.float64, device=full["dev"])
    ops.grad(L.LOSS_TRPO, th32, (4, H, H, 1), 1e-6, b, g, out2)
    o2 = out2.cpu().numpy()
    assert abs(o2[0] - o[0]) < 1e-9 and abs(o2[1] - o[1]) < 1e-13 and abs(o2[2] - o[2]) < 1e-11, (o, o2)


def test_fvp_is_linear_symmetric_and_positive(full):
    ops, b, th32, dev = full["ops"], full["b"], full["th32"], full["dev"]
    Pn = full["dims"].P
    rng = np.random.RandomState(2)
    x, y = (torch.tensor(rng.randn(Pn).astype(np.float32).astype(np.float64), device=dev) for _ in range(2))

    def F(v):
        out = torch.zeros(Pn, dtype=torch.float64, device=dev)
        ops.fvp(th32, (4, H, H, 1), 1e-6, b, v, 1e-5, 1.0, out)
        return out
    Fx, Fy = F(x), F(y)
    z = (0.5 * x - 2.0 * y)
    z = z.float().double()                                                 # tangent is rounded to float32 in-kernel
    Fz = F(z)
    lin = 0.5 * Fx - 2.0 * Fy
    assert float((Fz - lin).abs().max()) < 2e-5 * float(lin.abs().max())  # linearity
    sym = abs(float(x @ Fy) - float(y @ Fx))
    assert sym < 1e-5 * (abs(float(x @ Fy)) + 1e-12) + 1e-9                # symmetry
    assert float(x @ Fx) > 0 and float(y @ Fy) > 0                         # positive definite (+ reg)
    out2 = F(x)
    assert torch.equal(out2, Fx)                                           # deterministic (fixed-order reductions)


def test_gradient_matches_directional_derivative_of_the_loss(full):
    L, ops, b, th32, dev = full["L"], full["ops"], full["b"], full["th32"], full["dev"]
    Pn = full["dims"].P
    dd = (4, H, H, 1)
    g = torch.zeros(Pn, dtype=torch.float64, device=dev)
    ops.grad(L.LOSS_VPG, th32, dd, 1e-6, b, g)
    d = torch.tensor(np.random.RandomState(3).randn(Pn), dtype=torch.float64, device=dev)
    d = d / d.norm()
    out = torch.zeros(3, dtype=torch.float64, device=dev)
    eps = 2e-3
    vals = []
    for sgn in (+1.0, -1.0):
        thp = (th32.double() + sgn * eps * d).float()
        ops.loss_kl(L.LOSS_VPG, thp, dd, 1e-6, b, out)
        vals.append(float(out[0]))
    fd = (vals[0] - vals[1]) / (2 * eps)
    assert abs(fd - float(g @ d)) < 2e-3 * abs(float(g @ d)) + 1e-6, (fd, float(g @ d))


def test_rollout_is_deterministic_and_shard_invariant(full):
    """Same (seed, iter) -> identical bits; lanes generated as two half-size shards with lane0 offsets (what two GPUs
    do) are bit-identical to the single-GPU rollout: results do not depend on the number of GPUs."""
    L, ops, b, th32, dev = full["L"], full["ops"], full["b"], full["th32"], full["dev"]
    n = 4096
    ref = ops.LaneBatch(4, 1, n, 64, dev)
    ops.rollout(L.ENV_CARTPOLE, th32, H, H, 1e-6, ref, 64, None, None, 5, 9, 0)
    again = ops.LaneBatch(4, 1, n, 64, dev)
    ops.rollout(L.ENV_CARTPOLE, th32, H, H, 1e-6, again, 64, None, None, 5, 9, 0)
    halves = []
    for r in range(2):
        hb = ops.LaneBatch(4, 1, n // 2, 64, dev)
        ops.rollout(L.ENV_CARTPOLE, th32, H, H, 1e-6, hb, 64, None, None, 5, 9, r * (n // 2))
        halves.append(hb)
    for k in ("obs", "act", "mean", "rew", "flags"):
        assert torch.equal(getattr(ref, k), getattr(again, k)), k
        cat = torch.cat([getattr(halves[0], k), getattr(halves[1], k)], dim=-1)
        assert torch.equal(getattr(ref, k), cat), k
    other = ops.LaneBatch(4, 1, n, 64, dev)
    ops.rollout(L.ENV_CARTPOLE, th32, H, H, 1e-6, other, 64, None, None, 5, 10, 0)      # next iteration: new noise
    assert not torch.equal(ref.act, other.act)


def test_gradient_and_fisher_product_match_f64_kernels(full):
    """float32 TRPO gradient and cached Fisher product at cfg2 size against update_f64 (pinned to the float64 oracle by
    tests/test_gpu_multitile.py), in relative norm: ~26 000 tiles per pass, every CTA loops hundreds of times.  Measured
    on one B200: see DESIGN.md §5."""
    from test_gpu_multitile import TOL, _f32_vs_f64
    L, ops, b, th32 = full["L"], full["ops"], full["b"], full["th32"]
    x = np.random.RandomState(4).randn(full["dims"].P).astype(np.float32).astype(np.float64)
    err_g, err_H = _f32_vs_f64(ops, L, b, (4, H, H, 1), th32, x)
    print("\ncfg2: grad err %.3e  fvp err %.3e" % (err_g, err_H))
    assert err_g <= TOL["grad"] and err_H <= TOL["fvp"], (err_g, err_H)


def test_lfb_gram_and_fit_match_host_float64(full):
    """LinearFeatureBaseline normal equations over all 13.1 M samples against a float64 Gram accumulated on the host in
    chunks, and the device solve's predictions against the host's lstsq on that Gram."""
    from oracle import sampler as S
    ops, b, dev = full["ops"], full["b"], full["dev"]
    d1 = 2 * 4 + 5
    gram = torch.empty((d1 * (d1 + 1) // 2,), dtype=torch.float64, device=dev)
    ops.lfb_gram(b, gram)
    obs = b.obs.cpu().numpy().reshape(4, -1)
    ts = b.tstep.cpu().view(torch.int16).numpy().view(np.uint16).reshape(-1)
    ret = b.ret.cpu().numpy().reshape(-1)
    G = np.zeros((d1, d1))
    step = 1 << 20
    for i in range(0, N * T, step):
        F = np.concatenate([S.lfb_features_lanes(obs[:, i:i + step, None], ts[i:i + step, None])[:, :, 0],
                            ret[None, i:i + step].astype(np.float64)], axis=0)
        G += F @ F.T
    iu = np.triu_indices(d1)
    np.testing.assert_allclose(gram.cpu().numpy(), G[iu], rtol=2e-6, atol=1e-6 * np.abs(G).max())
    w_dev = torch.empty((d1 - 1,), dtype=torch.float64, device=dev)
    info = torch.zeros((3,), dtype=torch.float64, device=dev)
    ops.lfb_solve(4, gram, 1e-5, w_dev, info)
    reg, _, ok = info.cpu().tolist()
    assert ok == 1.0
    w_ref = S.lfb_fit_normal(G[:-1, :-1], G[:-1, -1], reg)
    sel = np.random.RandomState(0).choice(N * T, 1 << 20, replace=False)
    Fs = S.lfb_features_lanes(obs[:, sel, None], ts[sel, None])[:, :, 0].T
    pred, pred_ref = Fs @ w_dev.cpu().numpy(), Fs @ w_ref
    # Cholesky (device) and lstsq (host) on the same ill-conditioned d = 12 system: agree to 1e-3 of the prediction range
    assert np.abs(pred - pred_ref).max() <= 1e-3 * np.abs(pred_ref).max()
