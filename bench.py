"""bench.py -- env-steps/s of one full BatchPolopt iteration (rollout + process_samples + policy update) on B200.

Workload (BASELINE.json configs[1]): CartPoleEnv, 65 536 lanes per GPU, horizon 200, VPG + LinearFeatureBaseline,
GaussianMLPPolicy(32,32).  One "step" = one training iteration = N*T env steps.
  value  : device-resident iteration (policy parameters already in HBM), CUDA-event timed, max over ranks.
  e2e    : the same iteration through the plugin API with HOST parameter buffers: policy.set_param_values(host) ->
           algo.train_itr() -> policy.get_param_values() (+ the logged statistics and the baseline normal equations
           read back), host<->device copies inside the timed region.
  --impl reference : the reference's CPU sampler structure (oracle/cpu_sampler.py: per-path Python rollouts in a
           process pool over all host cores + NumPy update) on a bounded sample of the same workload.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True      # the benchmark leaves the source tree as it found it (it may be read-only)

WORKLOADS = {
    # name: (env, algo, lanes/GPU, horizon, hidden, alg bytes per env step (SURVEY 8d: 4*(O+3A+1)+1))
    "cartpole_vpg_65536x200": ("cartpole", "vpg", 65536, 200, 32, 33),
    "pendulum_vpg_262144x200": ("pendulum", "vpg", 262144, 200, 32, 29),
    "swimmer_trpo_16384x500": ("swimmer", "trpo", 16384, 500, 32, 81),
    "hopper_trpo_4096x500": ("hopper", "trpo", 4096, 500, 64, 121),
    "point_trpo_65536x100": ("point", "trpo", 65536, 100, 32, 37),
}


def make_env(name):
    from rllab_b200.envs.normalized_env import normalize
    if name == "cartpole":
        from rllab_b200.envs.box2d.cartpole_env import CartpoleEnv
        return normalize(CartpoleEnv())
    if name == "cartpole_swingup":
        from rllab_b200.envs.box2d.cartpole_swingup_env import CartpoleSwingupEnv
        return normalize(CartpoleSwingupEnv())
    if name == "double_pendulum":
        from rllab_b200.envs.box2d.double_pendulum_env import DoublePendulumEnv
        return normalize(DoublePendulumEnv())
    if name == "pendulum":
        from rllab_b200.envs.gym_env import GymEnv
        return normalize(GymEnv("Pendulum-v0"))
    if name == "point":
        from rllab_b200.envs.point_env import PointEnv
        return normalize(PointEnv())
    if name == "swimmer":
        from rllab_b200.envs.mujoco.swimmer_env import SwimmerEnv
        return normalize(SwimmerEnv())
    if name == "hopper":
        from rllab_b200.envs.mujoco.hopper_env import HopperEnv
        return normalize(HopperEnv())
    raise ValueError(name)


class ClockSampler(object):
    """nvidia-smi clocks / throttle reasons sampled during the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.proc = None
        self.idx = gpu_index
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(gpu_index)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["nvidia-smi unavailable"])
        time.sleep(0.05)
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except Exception:
            self.proc.kill()
            out = ""
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in out.strip().splitlines():
            f = [x.strip() for x in line.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1])), mx.append(float(f[2]))
            except ValueError:
                continue
            for nme, v in zip(names, f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(nme)
        return dict(sm_mhz=(statistics.median(sm) if sm else None), sm_max_mhz=(max(mx) if mx else None),
                    reasons=sorted(reasons), samples=len(sm))


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            d = json.load(open(p))
            return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, sustained copy)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def cpu_arm(workload, steps, warmup, cores=None, sample_steps=None, seconds_budget=20.0):
    """Reference CPU path (port): returns (env-steps/s, info)."""
    import numpy as np
    from oracle import cpu_sampler as C, policy as P, envs as E
    env_name, algo, lanes, T, hidden, _ = WORKLOADS[workload]
    cores = cores or os.cpu_count() or 1
    e = E.make(env_name)
    dims = P.Dims(e.O, (hidden, hidden), e.A)
    theta = P.init_params(dims, np.random.RandomState(1))
    sampler = C.CpuSampler(env_name, dims, cores, seed=1)
    # size the bounded sample: one short calibration iteration, then ~seconds_budget/(steps+warmup) per step
    if sample_steps is None:
        th, co, ad, ns, sec, _ = C.run_iteration(sampler, theta, None, dims, algo, 2000 * cores, T)
        rate = ns / max(sec, 1e-6)
        per_step = max(2.0, seconds_budget / max(1, steps + warmup))
        sample_steps = int(max(2000 * cores, min(rate * per_step, lanes * T)))
    coeffs, adam = None, None
    times, counts = [], []
    for i in range(warmup + steps):
        theta, coeffs, adam, ns, sec, avg_ret = C.run_iteration(sampler, theta, coeffs, dims, algo, sample_steps, T, adam)
        if i >= warmup:
            times.append(sec), counts.append(ns)
    sampler.close()
    value = sum(counts) / sum(times)
    info = dict(value=value, unit="env-steps/s", cores=cores, kind="port",
                sample="%d iterations of >=%d env steps each (whole paths, max_path_length %d) of %s; "
                       "per-path Python rollouts in %d worker processes + NumPy %s update (oracle/cpu_sampler.py)" %
                       (steps, sample_steps, T, workload, cores, algo.upper()))
    return value, info, sum(times) / len(times) * 1e3


def dump_outputs(out_dir, algo, policy, baseline, lanes_budget_bytes=32 << 20):
    """--dump-outputs: what the last timed iteration hands back to its caller, one .npy file per array in out_dir.
      policy_params, baseline_coeffs  float64, after that iteration's update and baseline fit
      stat_<key>                      float64 scalars, the iteration's logger.record_tabular table
      observations, actions, means    float32, [dim][T][lane] as the device holds them, for a fixed, seeded sample of
      rewards, advantages, returns,   this rank's lanes (at most lanes_budget_bytes in all); flags are the FLAG_* bits
      baselines, flags                of include/b200rl.h, masked samples included
      lanes                           float64, global index of each sampled lane
    The inputs of the iteration follow from the arguments and fixed seeds alone, so two builds run with the same
    arguments can be compared file by file."""
    import numpy as np
    import torch
    from rllab_b200.misc import logger
    b = algo.sampler.batch
    out = dict(policy_params=np.asarray(policy.get_param_values(), dtype=np.float64))
    coeffs = baseline.get_param_values()
    if coeffs is not None:
        out["baseline_coeffs"] = np.asarray(coeffs, dtype=np.float64)
    for k, v in logger.get_last_table().items():
        if isinstance(v, (int, float, np.number)):
            out["stat_" + k] = np.float64(v)
    planes = dict(observations=b.obs, actions=b.act, means=b.mean, rewards=b.rew, advantages=b.adv, returns=b.ret,
                  baselines=b.base, flags=b.flags)
    per_lane = 4 * b.T * sum(t.numel() // (b.T * b.N) for t in planes.values())
    n_sample = min(b.N, max(1, lanes_budget_bytes // per_lane))
    idx = np.sort(np.random.RandomState(0).choice(b.N, n_sample, replace=False))
    sel = torch.as_tensor(idx, device=b.device)
    for name, t in planes.items():
        out[name] = t.index_select(t.dim() - 1, sel).cpu().numpy().astype(np.float32)
    out["lanes"] = (idx + algo.sampler.lane0).astype(np.float64)
    assert sum(a.nbytes for a in out.values()) <= 64 << 20
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="cartpole_vpg_65536x200", choices=sorted(WORKLOADS))
    ap.add_argument("--lanes", type=int, default=None, help="lanes per GPU (default: the workload's)")
    ap.add_argument("--horizon", type=int, default=None)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the short TRPO workloads reported under extra.workloads")
    ap.add_argument("--cpu-seconds", type=float, default=15.0)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed iteration computed to DIR/<name>.npy (see dump_outputs)")
    ap.add_argument("--cpu-arm-json", action="store_true", help=argparse.SUPPRESS)   # internal: CPU leg in a clean process
    args = ap.parse_args()
    assert args.warmup >= 0 and args.steps >= 1
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    env_name, algo_name, lanes, T, hidden, alg_bytes = WORKLOADS[args.workload]
    lanes = args.lanes or lanes
    T = args.horizon or T

    if args.cpu_arm_json:
        # the cpu_baseline leg of the default run, executed in a fresh interpreter: its worker pool forks, and a fork
        # of a process that has initialised CUDA dies in the children as soon as one of them frees a device object
        _, info, _ = cpu_arm(args.workload, 2, 1, seconds_budget=args.cpu_seconds)
        print(json.dumps(info))
        return
    if args.impl == "reference":
        if rank != 0:
            return
        value, info, ms = cpu_arm(args.workload, args.steps, args.warmup, seconds_budget=90.0)
        line = dict(metric="env-steps/sec (full iteration: rollout + process_samples + %s update)" % algo_name.upper(),
                    value=value, unit="env-steps/s", n_gpus=args.gpus, steps=args.steps, warmup=args.warmup,
                    ms_per_step=ms, higher_is_better=True, scaling="weak", vs_baseline=None, dtype="f64",
                    data="synthetic", impl="reference",
                    config=dict(workload=args.workload, env=env_name, algo=algo_name, lanes_per_gpu=lanes, horizon=T,
                                hidden=[hidden, hidden], samples_per_step=lanes * T * args.gpus,
                                parallelism="host process pool (%d workers)" % info["cores"],
                                note="each step is a bounded sample of the workload (see cpu_baseline.sample)"),
                    cpu_baseline=info,
                    e2e=dict(value=value, unit="env-steps/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0),
                    gpu_launches=0)
        print(json.dumps(line))
        return

    import numpy as np
    import torch
    from rllab_b200 import _lib as L
    from rllab_b200 import ops
    from rllab_b200.misc import logger
    from rllab_b200.parallel import Comm

    L.load()
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    comm = Comm()
    logger.set_quiet(True)
    dev = torch.device("cuda", local_rank)

    def sync_all():
        comm.barrier()
        torch.cuda.synchronize()

    def build(workload, lanes_override=None, horizon_override=None, the_comm=comm, seed=1):
        from rllab_b200.algos.trpo import TRPO
        from rllab_b200.algos.vpg import VPG
        from rllab_b200.baselines.linear_feature_baseline import LinearFeatureBaseline
        from rllab_b200.policies.gaussian_mlp_policy import GaussianMLPPolicy
        env_n, algo_n, ln, hz, hid, _ = WORKLOADS[workload]
        ln, hz = lanes_override or ln, horizon_override or hz
        np.random.seed(1)
        env = make_env(env_n)
        policy = GaussianMLPPolicy(env.spec, hidden_sizes=(hid, hid), seed=1)
        baseline = LinearFeatureBaseline(env.spec)
        w = the_comm.world_size if the_comm.active else 1
        n_total = ln * w
        kw = dict(env=env, policy=policy, baseline=baseline, batch_size=n_total * hz, max_path_length=hz, n_itr=10 ** 9,
                  discount=0.99, sampler_args=dict(n_envs=n_total, seed=seed, comm=the_comm))
        algo = VPG(**kw) if algo_n == "vpg" else TRPO(step_size=0.01, **kw)
        algo.start_worker()
        algo.init_opt()
        return algo, policy, baseline, n_total * hz

    def run(algo, policy, n, itr0, e2e):
        """n iterations; returns elapsed ms on this rank (CUDA events on the launching stream)."""
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        host_theta = policy.get_param_values()
        sync_all()
        ev0.record()
        for i in range(n):
            if e2e:
                policy.set_param_values(host_theta)            # H2D: P float64 from host memory
            algo.train_itr(itr0 + i)
            if e2e:
                host_theta = policy.get_param_values()         # D2H: P float64
        ev1.record()
        sync_all()
        return ev0.elapsed_time(ev1)

    def max_over_ranks(*vals):
        t = torch.tensor(list(vals), dtype=torch.float64, device=dev)
        comm.all_reduce_max(t)
        return [float(x) for x in t.cpu().numpy()]

    algo, policy, baseline, steps_per_iter = build(args.workload, args.lanes, args.horizon)
    itr = 0
    run(algo, policy, args.warmup, itr, False)
    itr += args.warmup
    clocks = ClockSampler(local_rank) if rank == 0 else None
    k0, c0, x0 = L.kernel_launches(), comm.n_collectives, comm.n_peer_exchanges
    ms_dev = run(algo, policy, args.steps, itr, False)
    launches = (L.kernel_launches() - k0) / args.steps
    collectives = (comm.n_collectives - c0) / args.steps            # NCCL collectives on the iteration's critical path
    peer_exchanges = (comm.n_peer_exchanges - x0) / args.steps      # peer-memory exchanges (fused or stand-alone kernels)
    itr += args.steps
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, algo, policy, baseline)
    d2h0 = ops.PendingHost.bytes_total
    ms_e2e = run(algo, policy, args.steps, itr, True)
    d2h_stats = (ops.PendingHost.bytes_total - d2h0) / args.steps    # statistics / loss triples read back per iteration
    itr += args.steps
    clk = clocks.stop() if clocks else None
    ms_dev, ms_e2e = max_over_ranks(ms_dev, ms_e2e)

    # ---- replicas must stay bit-identical: every rank applies the same update to the same all-reduced vectors
    theta_dev = policy.theta64
    replicas_identical = True
    if comm.active:
        gathered = [torch.empty_like(theta_dev) for _ in range(world)]
        comm.dist.all_gather(gathered, theta_dev)
        replicas_identical = all(bool(torch.equal(gathered[0], g)) for g in gathered)
        assert replicas_identical, "policy parameters differ across ranks"
        assert comm.peer_timeouts() == 0, "a peer-memory collective timed out"

    # ---- rank-count invariance on a small problem: the sharded run of this job reproduces, on every rank, the
    # single-process run of the same total lanes (Philox is keyed by the GLOBAL lane; reductions are float64, rank order)
    shard_check = None
    if comm.active:
        class _Solo(Comm):                                   # world-size-1 communicator inside this process
            def __init__(self):
                self.world_size, self.rank, self.local_rank, self.active = 1, 0, local_rank, False
                self._gather_bufs, self.n_collectives, self._owns_group = {}, 0, False
                self.peer, self.n_peer_exchanges, self._windows = False, 0, None
        small = "cartpole_vpg_65536x200"
        a_sh, p_sh, _, _ = build(small, 1024, 50, comm, seed=5)
        a_solo, p_solo, _, _ = build(small, 1024 * world, 50, _Solo(), seed=5)
        for i in range(3):
            a_sh.train_itr(i)
            a_solo.train_itr(i)
        torch.cuda.synchronize()
        t_sh, t_solo = p_sh.get_param_values(), p_solo.get_param_values()
        rel = float(np.max(np.abs(t_sh - t_solo)) / np.max(np.abs(t_solo)))
        rel = max_over_ranks(rel)[0]
        shard_check = dict(workload="cartpole VPG, %d lanes x 50 steps, 3 iterations" % (1024 * world),
                           max_rel_diff_vs_single_process=rel)
        # rollout, GAE scan, loss/KL, gradient: per-tile float32 partials over the same sample groups (shards are whole
        # tiles), float64 above -> identical up to float64 summation order.  The baseline normal equations accumulate
        # float32 inside one thread's ~170 samples, and that grouping depends on the shard size: 1e-7 relative in the
        # baseline weights, ~1e-9 in theta after three Adam steps.
        assert rel < 1e-7, "sharded run differs from the single-process run: %g" % rel

    # ---- per-kernel timing of the same iteration (CUDA events around each library call), for the rooflines
    env_name, algo_name, lanes, T, hidden, alg_bytes = WORKLOADS[args.workload]
    lanes, T = args.lanes or lanes, args.horizon or T
    b = algo.sampler.batch
    dims = policy.dims

    def timed(fn, reps=5):
        fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / reps

    # FP32 roofline of this box, measured here: 16 independent fma.rn.f32x2 chains per thread, no memory traffic
    sink = torch.zeros(4, dtype=torch.float32, device=dev)
    import ctypes
    fma = ctypes.c_longlong(0)
    def _ffma():
        L.call("b200rl_bench_ffma2", 4096, L.ptr(sink), ctypes.byref(fma), ctypes.c_void_p(torch.cuda.current_stream().cuda_stream))
    ms_ffma = timed(_ffma, reps=3)
    fp32_peak = 2.0 * fma.value / (ms_ffma * 1e-3) / 1e12         # TFLOP/s (1 FMA = 2 flop)
    hbm_peak, hbm_src = measured_peaks()

    g = torch.zeros(policy.n_params, dtype=torch.float64, device=dev)
    out3 = torch.zeros(3, dtype=torch.float64, device=dev)
    loss_kind = L.LOSS_VPG if algo_name == "vpg" else L.LOSS_TRPO
    O, A, h = policy.obs_dim, policy.action_dim, hidden
    samp_bytes = 4 * (O + 3 * A + 1)
    F = 2.0 * (O * h + h * h + h * A)                               # flops of one policy forward
    n_valid = float(b.count.cpu()[0]) if b.masked else float(b.B_global)
    kern = {}
    kern["rollout"] = dict(ms=timed(lambda: ops.rollout(algo.sampler.env_kind, policy.theta32, hidden, hidden,
                                                        policy.min_std, b, T, None, None, 1, 12345, algo.sampler.lane0)),
                           bytes=alg_bytes * b.B, flops=F * b.B, per_iter=1, bound="fp32_issue")
    w = baseline.device_weights(b.O, dev)
    drop = bool(algo.whole_paths)
    kern["process_samples"] = dict(ms=timed(lambda: ops.process_samples(b, w, 0.99, 1.0, drop_cut_paths=drop)),
                                   bytes=(4 * O + 4 + 1 + 2 + 12) * b.B, flops=0.0, per_iter=1, bound="hbm")
    gram = torch.empty_like(b.gram)
    kern["lfb_gram"] = dict(ms=timed(lambda: ops.lfb_gram(b, gram)), bytes=(4 * O + 2 + 4 + 1) * b.B, flops=0.0,
                            per_iter=1, bound="hbm")
    kern["loss_kl"] = dict(ms=timed(lambda: ops.loss_kl(loss_kind, policy.theta32, dims, policy.min_std, b, out3)),
                           bytes=samp_bytes * b.B, flops=F * b.B, per_iter=1 if algo_name == "vpg" else 2,
                           bound="fp32_issue")
    kern["grad"] = dict(ms=timed(lambda: ops.grad(loss_kind, policy.theta32, dims, policy.min_std, b, g)),
                        bytes=samp_bytes * b.B, flops=(2 * F + 2.0 * (h * A + h * h)) * b.B, per_iter=1,
                        bound="fp32_issue")
    if algo_name == "trpo":
        x = torch.randn(policy.n_params, dtype=torch.float64, device=dev)
        Hx = torch.zeros_like(x)
        hc = b.hcache(h, h)
        ops.grad(loss_kind, policy.theta32, dims, policy.min_std, b, g, None, hc)
        fvp_flops = (2.0 * O * h + 4.0 * h * h + 4.0 * h * A + 2.0 * (h * A + h * h) + F) * b.B
        kern["fvp"] = dict(ms=timed(lambda: ops.fvp(policy.theta32, dims, policy.min_std, b, x, 1e-5, 1.0, Hx, hc)),
                           bytes=(4 * O + 8 * h) * b.B, flops=fvp_flops, per_iter=11, bound="fp32_issue")
    for k, v in kern.items():
        v["GBps"] = v["bytes"] / (v["ms"] * 1e-3) / 1e9
        v["TFLOPs"] = v["flops"] / (v["ms"] * 1e-3) / 1e12
        v["frac"] = (v["GBps"] / hbm_peak) if v["bound"] == "hbm" else (v["TFLOPs"] / fp32_peak)
        v["share_of_step"] = v["ms"] * v["per_iter"] / (ms_dev / args.steps)
    dom = max(kern, key=lambda k: kern[k]["ms"] * kern[k]["per_iter"])
    # dram bytes per launch from the ncu --set full capture of the shipped build (profiles/r02_traffic.json, written by
    # scripts/ncu_traffic.py from the committed capture); only quoted for the profiled geometry
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "r02_traffic.json")
    if os.path.exists(tpath) and args.lanes is None and args.horizon is None:
        try:
            traffic = json.load(open(tpath)).get(args.workload, {}).get(dom)
        except Exception:
            traffic = None
    kd = kern[dom]
    if kd["bound"] == "hbm":
        roofline = dict(bound="hbm", kernel=dom, achieved=kd["GBps"], peak=hbm_peak, unit="GB/s", frac=kd["frac"],
                        traffic=traffic, peak_source=hbm_src)
    else:
        roofline = dict(bound="fp32_issue", kernel=dom, achieved=kd["TFLOPs"], peak=fp32_peak, unit="TFLOP/s",
                        frac=kd["frac"], traffic=traffic,
                        peak_source="measured in this run: b200rl_bench_ffma2 (independent fma.rn.f32x2 chains, no memory)",
                        algorithmic_flops_per_launch=kd["flops"], algorithmic_bytes_per_launch=kd["bytes"],
                        hbm_GBps=kd["GBps"], hbm_frac=kd["GBps"] / hbm_peak,
                        note="the policy passes are bound by FP32 / instruction issue (%.0f flop per byte), not by HBM; "
                             "the HBM-bound kernel of the step is process_samples, reported under roofline_hbm" %
                             (kd["flops"] / max(kd["bytes"], 1)))
    kp = kern["process_samples"]
    roofline_hbm = dict(bound="hbm", kernel="process_samples", achieved=kp["GBps"], peak=hbm_peak, unit="GB/s",
                        frac=kp["frac"], peak_source=hbm_src, algorithmic_bytes_per_launch=kp["bytes"],
                        launch_ms=kp["ms"])

    # ---- the other BASELINE configs that fit one GPU, a few iterations each (TRPO workloads: cfg3, cfg4 share)
    extra = {}
    if args.workload == "cartpole_vpg_65536x200" and not args.no_extra and args.lanes is None:
        for wl in ("swimmer_trpo_16384x500", "hopper_trpo_4096x500"):
            a2, p2, _, spi = build(wl)
            run(a2, p2, 3, 0, False)
            k1 = L.kernel_launches()
            ms2 = run(a2, p2, 3, 3, False)
            l2 = (L.kernel_launches() - k1) / 3
            ms2 = max_over_ranks(ms2)[0]
            extra[wl] = dict(ms_per_step=ms2 / 3, value=spi * 3 / (ms2 * 1e-3), unit="env-steps/s", steps=3, warmup=3,
                             gpu_launches=l2, samples_per_step=spi,
                             AverageReturn=a2.sampler.stats.get("AverageReturn"),
                             backtrack_iters=a2.optimizer.last_info.get("n_iter"),
                             MeanKL=a2.optimizer.last_info.get("constraint_val"))
            a2.shutdown_worker()
    if rank != 0:
        comm.close()
        return
    value = steps_per_iter * args.steps / (ms_dev * 1e-3)
    e2e_value = steps_per_iter * args.steps / (ms_e2e * 1e-3)
    P_ = policy.n_params
    line = dict(
        metric="env-steps/sec (full iteration: rollout + process_samples + %s update)" % algo_name.upper(),
        value=value, unit="env-steps/s", n_gpus=world, steps=args.steps, warmup=args.warmup,
        ms_per_step=ms_dev / args.steps, higher_is_better=True, scaling="weak", vs_baseline=None, dtype="f32",
        data="synthetic", impl="b200",
        config=dict(workload=args.workload, env=env_name, algo=algo_name, lanes_per_gpu=lanes, horizon=T,
                    hidden=[hidden, hidden], samples_per_step=steps_per_iter, parallelism="lanes sharded x%d" % world,
                    whole_paths=bool(algo.whole_paths), valid_samples_per_step=n_valid,
                    l2="trajectory buffers (%.0f MB/GPU) exceed the 126 MB L2" % (b.B * (alg_bytes + 14) / 1e6)),
        e2e=dict(value=e2e_value, unit="env-steps/s", ms_per_step=ms_e2e / args.steps,
                 h2d_bytes_per_step=8 * P_, d2h_bytes_per_step=8 * P_ + d2h_stats),
        gpu_launches=launches, collectives_per_step=collectives, peer_exchanges_per_step=peer_exchanges,
        transport=("peer-memory windows over NVLink (csrc/peer.cuh)" if comm.peer else
                   ("NCCL all-gather + rank-order fold" if comm.active else "single GPU")),
        clocks=clk, roofline=roofline,
        roofline_hbm=roofline_hbm, fp32_peak_tflops=fp32_peak,
        kernels={k: dict(ms=round(v["ms"], 4), GBps=round(v["GBps"], 1), TFLOPs=round(v["TFLOPs"], 2), bound=v["bound"],
                         frac=round(v["frac"], 4), per_iter=v["per_iter"], share_of_step=round(v["share_of_step"], 3))
                 for k, v in kern.items()},
        stats=dict(AverageReturn=algo.sampler.stats.get("AverageReturn"), NumTrajs=algo.sampler.stats.get("NumTrajs")),
        replicas_identical=replicas_identical, shard_check=shard_check,
        extra=dict(workloads=extra),
    )
    if env_name in ("swimmer", "hopper") and not args.no_cpu_baseline:
        # the planar-chain oracle is a slow float64 checker (tens of ms per scalar env step), not a CPU implementation
        # worth timing; the CPU baseline is reported for the classic-control workloads only.
        line["cpu_baseline"] = None
    elif world == 1 and not args.no_cpu_baseline:
        try:
            out = subprocess.run([sys.executable, os.path.abspath(__file__), "--cpu-arm-json", "--workload", args.workload,
                                  "--cpu-seconds", str(args.cpu_seconds)], capture_output=True, text=True, timeout=600,
                                 env=dict(os.environ, CUDA_VISIBLE_DEVICES=""))
            line["cpu_baseline"] = json.loads(out.stdout.strip().splitlines()[-1])
        except Exception as exc:                                            # noqa: BLE001
            line["cpu_baseline"] = dict(value=None, unit="env-steps/s", kind="port", error=repr(exc)[:200])
    print(json.dumps(line))
    comm.close()


if __name__ == "__main__":
    main()
