"""GPU: the update passes at batch sizes where every persistent CTA walks many 128-sample tiles, against the float64
oracle (oracle/policy.py) on the valid samples.

The tcgen05 kernels (update_umma.cu, update_umma32.cu), the FFMA kernels (update_tile.cu, update_gemm.cu) and the
float64 parity kernel (update_f64.cu) are persistent: each CTA strides over the tiles and carries state from one tile
to the next -- the mbarrier phase, float32 Gram accumulators flushed to float64 every 8 tiles, the L2 prefetch of the
next tile, the TMEM and shared-memory stage rows.  At the sizes of test_gpu_kernels.py no CTA reaches its second tile;
here every one does.

Tolerances are relative norms, ||device - oracle|| / ||oracle||.  Each float32 gradient and Fisher-product comparison
also computes the oracle with one tile's valid samples left out and requires its tolerance to be at most a tenth of the
change that makes: a kernel that drops or double-counts one tile fails the test, and a tolerance too loose to see that
fails it as well."""
import ctypes

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from oracle import policy as P          # noqa: E402

TILE = 128
NETS = [(O, A, H) for H in (32, 64) for (O, A) in ((2, 2), (3, 1), (4, 1), (6, 1), (13, 2), (20, 3))]
REG = 1e-5
# float32 passes against the float64 oracle, relative norm.  Largest errors measured on one B200 (1000 W) over every
# case of this file: loss 7.9e-5, gradient 5.7e-6, Fisher product 1.8e-6; smallest one-tile changes: gradient 4.4e-3,
# Fisher product 4.0e-5.
TOL = dict(loss=1e-4, grad=1e-4, fvp=3e-6)
MARGIN = 10.0           # a tolerance must be this many times smaller than the effect of one missing tile


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from rllab_b200 import _lib
    _lib.load()
    return torch.device("cuda:0")


def _ops():
    from rllab_b200 import ops
    return ops


def _L():
    from rllab_b200 import _lib
    return _lib


def _sms():
    L = _L()
    n = ctypes.c_int(0)
    L.check(L.load().b200rl_device_sms(ctypes.byref(n)), "b200rl_device_sms")
    return n.value


def _rel(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return float(np.linalg.norm(a - b) / np.linalg.norm(b))


class Multi(object):
    """A synthetic batch of N = 20*sms + 41 lanes x T = 127 steps.  On 148 SMs: B = 381 127 samples, 2 978 tiles, the
    last one 71 samples long.  B is odd (the activation cache takes its scalar path); no grid size divides the tile
    count; a 64-wide CTA (one per SM) runs 20-21 tiles and so crosses two float32->float64 flushes; a 32-wide CTA
    (two to four per SM) runs 5-10 tiles.

    obs ~ N(0,1) with the first and the last dimension scaled x30 (saturated tanh units); old_mean / act from
    b200rl_policy_get_actions at theta_old; adv ~ N(0,1); FLAG_MASKED on ~10 % of the samples at random and on three
    whole tiles, or -- with `valid_tiles` -- on every sample outside those tiles."""

    def __init__(self, dev, O, A, H, min_std=1e-6, low_ls=False, valid_tiles=None, seed=0):
        ops, L = _ops(), _L()
        self.ops, self.L, self.dev = ops, L, dev
        self.O, self.A, self.H, self.min_std = O, A, H, min_std
        self.N, self.T = 20 * _sms() + 41, 127
        B = self.B = self.N * self.T
        self.ntiles = -(-B // TILE)
        self.dims = P.Dims(O, (H, H), A)
        self.dd = (O, H, H, A)
        self.ols = self.dims.P - A
        rng = self.rng = np.random.RandomState(1000 * O + 10 * H + A + seed)
        theta = P.init_params(self.dims, rng) + rng.randn(self.dims.P) * 0.05
        theta[self.ols:] = -0.5 + 0.1 * np.arange(A)
        if low_ls:
            theta[self.ols] = np.log(min_std) - 1.0          # clamped to log(min_std): per dimension
        self.th32 = torch.tensor(theta, dtype=torch.float32, device=dev)
        self.theta = self.th32.cpu().numpy().astype(np.float64)
        obs = rng.randn(O, B).astype(np.float32)
        obs[0] *= 30.0
        obs[-1] *= 30.0
        b = self.b = ops.LaneBatch(O, A, self.N, self.T, dev)
        b.obs.copy_(torch.from_numpy(obs.reshape(O, self.T, self.N)))
        eps = torch.from_numpy(rng.randn(A, B).astype(np.float32)).to(dev)
        ops.policy_get_actions(self.th32, O, H, H, A, min_std, b.obs, B, eps, 0, 0, 0, 0, b.act, b.mean, b.log_std)
        b.adv.copy_(torch.from_numpy(rng.randn(self.T, self.N).astype(np.float32)))
        tile = np.arange(B) // TILE
        if valid_tiles is None:
            masked = rng.rand(B) < 0.1
            masked |= np.isin(tile, [3, self.ntiles // 2, self.ntiles - 2])
        else:
            masked = ~np.isin(tile, valid_tiles)
        self.valid = ~masked
        b.flags.copy_(torch.from_numpy(np.where(masked, L.FLAG_MASKED, 0).astype(np.uint8).reshape(self.T, self.N)))
        b.masked = True
        b.count.fill_(float(self.valid.sum()))
        torch.cuda.synchronize()
        self.obs = obs.T.astype(np.float64)
        self.act = b.act.cpu().numpy().reshape(A, B).T.astype(np.float64)
        self.mean = b.mean.cpu().numpy().reshape(A, B).T.astype(np.float64)
        self.adv = b.adv.cpu().numpy().reshape(B).astype(np.float64)
        self.log_std = b.log_std.cpu().numpy().astype(np.float64)
        self.eps = eps.cpu().numpy().T.astype(np.float64)

    def batch(self, idx=None):
        """Oracle batch of the valid samples (of the samples `idx`, if given)."""
        keep = np.flatnonzero(self.valid) if idx is None else np.asarray(idx)
        return dict(obs=self.obs[keep], actions=self.act[keep], adv=self.adv[keep], old_mean=self.mean[keep],
                    old_log_std=self.log_std)

    def some_tiles(self, k, among=None):
        """k random complete tiles (from `among`, if given) that hold valid samples."""
        cand = np.arange(self.ntiles - 1) if among is None else np.asarray(among)
        cand = cand[[(t + 1) * TILE <= self.B and self.valid[t * TILE:(t + 1) * TILE].any() for t in cand]]
        return np.random.RandomState(7).choice(cand, min(k, cand.size), replace=False)

    def tile_idx(self, t):
        """valid samples of tile t"""
        idx = np.arange(t * TILE, min((t + 1) * TILE, self.B))
        return idx[self.valid[idx]]

    def m_l(self):
        """log_std block of the Fisher matrix: diagonal, zero where the min_std clamp is active."""
        ls = self.theta[self.ols:]
        s = np.exp(2.0 * ls)
        ml = 4.0 * s * (2.0 * s - 1e-8) / np.square(2.0 * s + 1e-8)
        return np.where(ls > np.log(self.min_std), ml, 0.0)


def _one_tile(m, f_all, n, fn, tiles):
    """Relative change of an oracle mean when one tile's samples are left out, smallest over `tiles`.  f_all: the mean
    over n valid samples; fn(batch): the same mean over another batch.  Without the n_t valid samples of tile t the
    mean is (n f_all - n_t f_t) / (n - n_t)."""
    drops = []
    for t in tiles:
        idx = m.tile_idx(t)
        f_minus = (n * np.asarray(f_all) - idx.size * np.asarray(fn(m.batch(idx)))) / (n - idx.size)
        drops.append(_rel(f_minus, f_all))
    return min(drops)


def _verdict(name, err, tol, drop=None, margin=True):
    """err within tol, and (drop given, margin) tol small enough to see one missing tile"""
    print("  %-24s err %.3e  tol %.0e  one tile %s" % (name, err, tol, "-" if drop is None else "%.3e" % drop))
    assert err <= tol, "%s: error %.3e above %.0e" % (name, err, tol)
    if drop is not None and margin:
        assert tol * MARGIN <= drop, "%s: tolerance %.0e cannot see one missing tile (%.3e)" % (name, tol, drop)


def _fvp_oracle(m, batch, x32):
    """Sample part of the Fisher product (x's log_std entries do not enter it) in float64."""
    xw = x32.copy()
    xw[m.ols:] = 0.0
    return P.fvp(m.theta, batch, xw, m.dims, 0.0, m.min_std)


def _diag_part(m, x):
    d = REG * x.copy()
    d[m.ols:] += m.m_l() * x[m.ols:]
    return d


def _device_fvp(m, x, ds, cache, tile_list=None, count=None):
    out = torch.zeros(m.dims.P, dtype=torch.float64, device=m.dev)
    xd = torch.tensor(x, dtype=torch.float64, device=m.dev)
    m.ops.fvp(m.th32, m.dd, m.min_std, m.b, xd, REG, ds, out, cache, tile_list, count)
    return out.cpu().numpy()


def _write_cache(m):
    hc = m.b.hcache(m.H, m.H)
    g = torch.zeros(m.dims.P, dtype=torch.float64, device=m.dev)
    m.ops.grad(m.L.LOSS_TRPO, m.th32, m.dd, m.min_std, m.b, g, None, hc)
    return hc




def _perturbed(m, seed=9):
    """theta_old + N(0, 0.02^2), rounded to the float32 the kernels read"""
    th32 = torch.tensor(m.theta + np.random.RandomState(seed).randn(m.dims.P) * 0.02, dtype=torch.float32,
                        device=m.dev)
    return th32, th32.cpu().numpy().astype(np.float64)


def _check_grad(m, name, th, th32, batch, tiles, h_cache=None):
    """float32 gradient pass (and its fused loss triple) at th against the oracle."""
    L = m.L
    kind = L.LOSS_TRPO if name == "trpo" else L.LOSS_VPG
    surr = P.surr_loss_trpo if name == "trpo" else P.surr_loss_vpg
    n = len(batch["adv"])
    g = torch.zeros(m.dims.P, dtype=torch.float64, device=m.dev)
    out = torch.zeros(3, dtype=torch.float64, device=m.dev)
    m.ops.grad(kind, th32, m.dd, m.min_std, m.b, g, out, h_cache)
    gn, og = g.cpu().numpy(), out.cpu().numpy()
    ref_loss = surr(th, batch, m.dims, m.min_std)
    mkl, xkl = P.kl_stats(th, batch, m.dims, m.min_std)
    ref_g = P.grad_surr(th, batch, m.dims, name, m.min_std)
    drop_l = _one_tile(m, ref_loss, n, lambda bt: surr(th, bt, m.dims, m.min_std), tiles)
    drop_g = _one_tile(m, ref_g, n, lambda bt: P.grad_surr(th, bt, m.dims, name, m.min_std), tiles)
    # the loss is a scalar: a tile whose terms average to the batch mean leaves it unchanged, so its one-tile change is
    # reported, and the tile-level check rests on the gradient and the Fisher product (vectors of P entries)
    _verdict(name + " grad: loss", _rel(og[0], ref_loss), TOL["loss"], drop_l, margin=False)
    _verdict(name + " grad", _rel(gn, ref_g), TOL["grad"], drop_g)
    # mean / max KL: averages of non-negative terms, checked per value as in test_gpu_kernels.py
    np.testing.assert_allclose(og[1], mkl, rtol=2e-5, atol=1e-8)
    np.testing.assert_allclose(og[2], xkl, rtol=1e-4, atol=1e-8)
    clamped = m.theta[m.ols:] <= np.log(m.min_std)
    assert (gn[m.ols:][clamped] == 0.0).all() and (ref_g[m.ols:][clamped] == 0.0).all()
    return ref_loss, mkl, xkl


def _check_fvp(m, batch, tiles, x, caches, ds_list=(1.0,), tile_list=None, count=None):
    """Fisher product at theta_old through each h_cache in `caches` (None: FFMA kernels, recomputed activations; a cache:
    tcgen05 kernels) at each diag_scale: Hx(ds) = sample part + ds (reg x + M_l x_l)."""
    x32 = x.astype(np.float32).astype(np.float64)          # the kernels read the tangent in float32
    S = _fvp_oracle(m, batch, x32)
    D = _diag_part(m, x)
    drop = _one_tile(m, S + D, len(batch["adv"]), lambda bt: _fvp_oracle(m, bt, x32) + D, tiles)
    clamped = np.flatnonzero(m.theta[m.ols:] <= np.log(m.min_std)) + m.ols
    for cache in caches:
        for ds in ds_list:
            Hx = _device_fvp(m, x, ds, cache, tile_list, count)
            ref = S + ds * D
            _verdict("fvp %s ds=%g" % ("ffma" if cache is None else "cached", ds), _rel(Hx, ref), TOL["fvp"], drop)
            # an entry at the clamp gets reg * x only (no M_l term, no sample part)
            np.testing.assert_allclose(Hx[clamped], ds * REG * x[clamped], rtol=1e-12, atol=0)


# ------------------------------------------------------------------------------------------- A + C: every net
CASES = [(O, A, H, False) for (O, A, H) in NETS] + [(O, A, H, True) for (O, A, H) in NETS if A >= 2]


@pytest.mark.parametrize("O,A,H,low_ls", CASES,
                         ids=["%d-%d-%d%s" % (O, A, H, "-lowstd" if lo else "") for (O, A, H, lo) in CASES])
def test_update_passes_match_oracle_multitile(dev, O, A, H, low_ls):
    """Every pass of every compiled net against the oracle: get_actions, loss/KL (TRPO, VPG), the gradient with its
    fused loss triple, the Fisher product through both kernel families at diag_scale 1, 0.25 and 0 (the split the
    ranks of a sharded job rely on, include/b200rl.h b200rl_fvp), and update_f64 modes 0, 1, 2.

    low_ls: min_std = 1e-3 and the first log_std entry below log(min_std).  The clamp is per dimension: that entry's
    gradient and Fisher entries must be the clamp's (zero; reg x), the others must not.  With a std of 1e-3 the TRPO
    ratio at perturbed parameters underflows, so that case runs VPG only."""
    min_std = 1e-3 if low_ls else 1e-6
    m = Multi(dev, O, A, H, min_std=min_std, low_ls=low_ls)
    ops, L = m.ops, m.L
    print("\n(%d,%d,%d)%s  B=%d tiles=%d valid=%d" % (O, A, H, " low log_std" if low_ls else "", m.B, m.ntiles,
                                                     m.valid.sum()))
    # get_actions against the oracle forward (every sample, masked ones included)
    mu, lsd = P.forward(m.theta, m.obs, m.dims, min_std)
    np.testing.assert_allclose(m.mean, mu, rtol=2e-5, atol=2e-6)
    np.testing.assert_allclose(m.act, mu + np.exp(lsd) * m.eps, rtol=2e-5, atol=2e-6)
    np.testing.assert_allclose(m.log_std, lsd, rtol=1e-6)

    batch = m.batch()
    tiles = m.some_tiles(4)
    names = ("vpg",) if low_ls else ("trpo", "vpg")
    out = torch.zeros(3, dtype=torch.float64, device=dev)
    if not low_ls:
        # theta_old: likelihood ratio 1 -> loss -mean(adv), KL 0
        ops.loss_kl(L.LOSS_TRPO, m.th32, m.dd, min_std, m.b, out)
        o = out.cpu().numpy()
        if H == 64:      # FFMA loss kernel: the summation order of get_actions, ratio exactly 1
            assert abs(o[0] + batch["adv"].mean()) < 1e-12 and abs(o[1]) < 1e-12 and abs(o[2]) < 1e-12, o
        else:            # tensor-core forward (3xTF32): get_actions' mean to ~1e-7
            assert abs(o[0] + batch["adv"].mean()) < 1e-7 and abs(o[1]) < 1e-10 and abs(o[2]) < 1e-8, o
    th2_32, th2 = _perturbed(m)
    for name in names:
        kind = L.LOSS_TRPO if name == "trpo" else L.LOSS_VPG
        ref_loss, mkl, xkl = _check_grad(m, name, th2, th2_32, batch, tiles)
        ops.loss_kl(kind, th2_32, m.dd, min_std, m.b, out)
        o = out.cpu().numpy()
        _verdict(name + " loss_kl", _rel(o[0], ref_loss), TOL["loss"])
        np.testing.assert_allclose(o[1], mkl, rtol=2e-5, atol=1e-8)
        np.testing.assert_allclose(o[2], xkl, rtol=1e-4, atol=1e-8)

    hc = _write_cache(m)
    x = np.random.RandomState(10).randn(m.dims.P)
    _check_fvp(m, batch, tiles, x, (None, hc), ds_list=(1.0, 0.25, 0.0))

    # float64 parity kernel (grid-stride loop over many passes): loss/KL and gradient at unrounded perturbed
    # parameters, Fisher product at theta_old
    th64 = m.theta + np.random.RandomState(4).randn(m.dims.P) * 0.02
    thd = torch.tensor(th64, dtype=torch.float64, device=dev)
    g = torch.zeros(m.dims.P, dtype=torch.float64, device=dev)
    for name in names:
        kind = L.LOSS_TRPO if name == "trpo" else L.LOSS_VPG
        ops.update_f64(0, kind, thd, m.dd, min_std, m.b, None, 0.0, 0.0, None, out)
        ref_loss = (P.surr_loss_trpo if name == "trpo" else P.surr_loss_vpg)(th64, batch, m.dims, min_std)
        mkl, xkl = P.kl_stats(th64, batch, m.dims, min_std)
        np.testing.assert_allclose(out.cpu().numpy(), [ref_loss, mkl, xkl], rtol=1e-9, atol=1e-13)
        ops.update_f64(1, kind, thd, m.dd, min_std, m.b, None, 0.0, 0.0, g, out)
        ref_g = P.grad_surr(th64, batch, m.dims, name, min_std)
        np.testing.assert_allclose(g.cpu().numpy(), ref_g, rtol=1e-8, atol=1e-12 * np.abs(ref_g).max())
    Hx = torch.zeros(m.dims.P, dtype=torch.float64, device=dev)
    th0 = torch.tensor(m.theta, dtype=torch.float64, device=dev)
    ops.update_f64(2, L.LOSS_TRPO, th0, m.dd, min_std, m.b, torch.tensor(x, dtype=torch.float64, device=dev), REG,
                   1.0, Hx, None)
    ref_Hx = P.fvp(m.theta, batch, x, m.dims, REG, min_std)
    np.testing.assert_allclose(Hx.cpu().numpy(), ref_Hx, rtol=1e-8, atol=1e-12 * np.abs(ref_Hx).max())


# ------------------------------------------------------------------------------------------- B: sparse valid tiles
@pytest.mark.parametrize("O,A,H", [(13, 2, 32), (6, 1, 64)])
def test_sparse_valid_tiles_match_oracle(dev, O, A, H):
    """Only the tiles k = 5 (mod 37) hold valid samples.  37 is coprime with every grid size, so the ~80 valid tiles
    fall on varied loop iterations of varied CTAs, and each carries ~1/80 of the result."""
    ntiles = -(-((20 * _sms() + 41) * 127) // TILE)
    keep = np.arange(5, ntiles, 37)
    m = Multi(dev, O, A, H, valid_tiles=keep)
    print("\n(%d,%d,%d) sparse: %d valid tiles of %d" % (O, A, H, keep.size, m.ntiles))
    batch = m.batch()
    tiles = m.some_tiles(4, keep)
    th2_32, th2 = _perturbed(m)
    _check_grad(m, "trpo", th2, th2_32, batch, tiles)
    hc = _write_cache(m)
    _check_fvp(m, batch, tiles, np.random.RandomState(3).randn(m.dims.P), (None, hc))


# ------------------------------------------------------------------------------------------- D: tile lists
@pytest.mark.parametrize("O,A,H", [(4, 1, 32), (20, 3, 64)])
def test_tile_list_fvp_matches_oracle(dev, O, A, H):
    """The sub-sampled Fisher product (subsample_factor < 1): a random 30 % of the tiles in shuffled order, with the
    partial last tile and the fully masked tiles among them.  count_valid is exact; both Fisher paths match the oracle
    on the valid samples of the listed tiles."""
    m = Multi(dev, O, A, H)
    rng = np.random.RandomState(21)
    pick = rng.choice(m.ntiles, int(0.3 * m.ntiles), replace=False)
    pick = np.union1d(pick, [3, m.ntiles // 2, m.ntiles - 2, m.ntiles - 1])
    rng.shuffle(pick)
    assert m.B % TILE != 0
    tl = torch.tensor(pick.astype(np.int32), device=dev)
    idx = np.concatenate([m.tile_idx(t) for t in pick])
    count = torch.zeros(1, dtype=torch.float64, device=dev)
    m.ops.count_valid(m.b, None, count)
    assert count.item() == float(m.valid.sum())
    m.ops.count_valid(m.b, tl, count)
    assert count.item() == float(idx.size)
    print("\n(%d,%d,%d) tile list: %d of %d tiles, %d valid samples" % (O, A, H, pick.size, m.ntiles, idx.size))
    hc = _write_cache(m)
    _check_fvp(m, m.batch(idx), m.some_tiles(4, pick), np.random.RandomState(5).randn(m.dims.P), (None, hc),
               tile_list=tl, count=count)


# ------------------------------------------------------------------------------------------- E: benchmark sizes
@pytest.mark.parametrize("env_name,hidden,N,T", [("swimmer", 32, 16384, 500), ("hopper", 64, 4096, 500)],
                         ids=["cfg3-swimmer", "cfg4-hopper"])
def test_benchmark_sizes_match_f64_kernels(dev, env_name, hidden, N, T):
    """cfg3 (Swimmer, (32,32), 16 384 x 500) and cfg4 (Hopper, (64,64), 4 096 x 500) as bench.py runs them: device
    rollout, process_samples with drop_cut_paths, centred advantages; float32 gradient and cached Fisher product at
    theta_old against update_f64 (which test_update_passes_match_oracle_multitile pins to the oracle), relative norm.
    Measured on one B200 (1000 W): gradient 4.1e-7 (both), Fisher product 9.1e-7 (cfg3) and 1.1e-6 (cfg4)."""
    from oracle import envs as E
    ops, L = _ops(), _L()
    env = E.make(env_name)
    dd = (env.O, hidden, hidden, env.A)
    dims = P.Dims(env.O, (hidden, hidden), env.A)
    theta = P.init_params(dims, np.random.RandomState(11))
    theta[-env.A:] = -0.5
    th32 = torch.tensor(theta, dtype=torch.float32, device=dev)
    b = ops.LaneBatch(env.O, env.A, N, T, dev)
    ops.rollout(L.ENV_KINDS[env_name], th32, hidden, hidden, 1e-6, b, T, None, None, 1, 3, 0)
    ops.process_samples(b, None, 0.99, 0.97, drop_cut_paths=True)
    ops.center_advantages(b, True, False)
    x = np.random.RandomState(2).randn(dims.P).astype(np.float32).astype(np.float64)
    err_g, err_H = _f32_vs_f64(ops, L, b, dd, th32, x)
    print("\n%s B=%d valid=%d" % (env_name, b.B, int(b.count.item())))
    _verdict("trpo grad vs f64", err_g, TOL["grad"])
    _verdict("fvp cached vs f64", err_H, TOL["fvp"])


def _f32_vs_f64(ops, L, b, dd, th32, x):
    """Relative-norm errors of the float32 TRPO gradient and cached Fisher product against update_f64 at th32; x is
    float32-representable, so both read the same tangent."""
    dev = th32.device
    Pn = th32.numel()
    th64 = th32.double()
    xd = torch.tensor(x, dtype=torch.float64, device=dev)
    ref_g, ref_H, g, Hx = (torch.zeros(Pn, dtype=torch.float64, device=dev) for _ in range(4))
    out = torch.zeros(3, dtype=torch.float64, device=dev)
    ops.update_f64(1, L.LOSS_TRPO, th64, dd, 1e-6, b, None, 0.0, 0.0, ref_g, out)
    ops.update_f64(2, L.LOSS_TRPO, th64, dd, 1e-6, b, xd, REG, 1.0, ref_H, None)
    hc = b.hcache(dd[1], dd[2])
    ops.grad(L.LOSS_TRPO, th32, dd, 1e-6, b, g, None, hc)
    ops.fvp(th32, dd, 1e-6, b, xd, REG, 1.0, Hx, hc)
    return _rel(g.cpu().numpy(), ref_g.cpu().numpy()), _rel(Hx.cpu().numpy(), ref_H.cpu().numpy())
