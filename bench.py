#!/usr/bin/env python
"""bench.py -- env-steps/s of the batched SMPL-humanoid stepper (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            (N>1: launched by torch.distributed.run)
    python bench.py --impl reference --gpus N --steps K --warmup W
    python bench.py --gpus 1 --steps K --warmup W --dump-outputs DIR   (+ what the last timed step returned, DIR/<name>.npy)

Workload (BASELINE.json configs[1], SURVEY.md 8d "Config 2"): 4 096 SMPL envs per GPU, env=speed, flat ground,
state_init=Default, self_obs_v=1 (obs 292), control_mode=uhc_pd (the reference's yaml default: stable PD), actions
a ~ clip(N(0, 0.0821^2), -1, 1) drawn on the device with manual_seed(0), in-stream autoreset of terminated/truncated
envs (episode_length 300).  One "step" = one env.step() of every env (15 physics substeps + obs/reward/flags) followed
by the masked reset launch.  Envs shard across ranks with no collective on the physics path ("scaling": "weak").

The reference arm (--impl reference) times the CPU fp64 oracle port of the same path (oracle/; the reference's physics
lives in the absent `mujoco` wheel, so there is no oracle/_ref) on all host cores, on a bounded sample of the workload.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

ENVS_PER_GPU = 4096
SIGMA = float(np.exp(-2.5))          # learning/simple_mlp.yaml:11-12 fixed log_std
B_ALG_BYTES = 2682                   # SURVEY.md 8d, cfg2: (223 read + 447.5 written) fp32 words per env-step
B_ALG_STALE_BYTES = 1208             # + (qpos,qvel) of the last forward pass written + read (quirk-Q1 parity carry)
WORKLOAD = "cfg2: 4096 SMPL envs/GPU, env=speed, uhc_pd (stable PD), obs_v1=292, 15 substeps @450Hz, autoreset"
# --workload: the headline (cfg2, default) and the other single-GPU shapes of BASELINE.json's configs (variants, not the bench line)
WORKLOADS = {
    "cfg2": dict(env="speed", robot="smpl_humanoid", overrides={}, envs=4096, balg=2682, desc=WORKLOAD),
    "cfg2-pd": dict(env="speed", robot="smpl_humanoid", overrides={"env.control_mode": "pd"}, envs=4096, balg=2682,
                    desc="cfg2 variant: explicit PD (control_mode=pd), 4096 SMPL envs/GPU"),
    "cfg2-v2": dict(env="speed", robot="smpl_humanoid", overrides={"env.self_obs_v": 2, "robot.create_vel_sensors": True}, envs=4096, balg=2958,
                    desc="cfg2 variant: self_obs_v=2 (obs 361), 4096 SMPL envs/GPU"),
    "cfg3": dict(env="reach", robot="smpl_humanoid", overrides={"env.self_obs_v": 2, "robot.create_vel_sensors": True}, envs=16384, balg=2974,
                 desc="cfg3: 16384 SMPL envs/GPU, env=reach, self_obs_v=2 (obs 361), uhc_pd"),
    "cfg4": dict(env="speed", robot="smpl_humanoid", overrides={"env.self_obs_v": 2, "robot.create_vel_sensors": True}, envs=8192, balg=2958 + 4 * (76 + 75) * 2,
                 motion=True,
                 desc="cfg4 shard: 8192 SMPL envs/GPU (65 536 on 8), obs_v2=361, per-step get_motion_state_intervaled gather of the reference pose "
                      "(synthetic clip tables, SURVEY 8d) + MoCap reset of finished envs from the gathered frame, uhc_pd"),
    "cfg5": dict(env="getup", robot="smplx_humanoid", overrides={}, envs=4096, balg=5698,
                 desc="cfg5 shard: 4096 SMPL-X (52 bodies) envs/GPU, env=getup (Fall init), obs_v1, uhc_pd"),
    "cfg2-selfcol": dict(env="speed", robot="smpl_humanoid", overrides={"env.self_collision": True}, envs=4096, balg=2682,
                         desc="cfg2 with cfg.env.self_collision: geom-geom contacts (capsule / sphere pairs, MuJoCo's filters) simulated as two-body rows"),
    "cfg2-shapes": dict(env="speed", robot="smpl_humanoid", overrides={}, envs=4096, balg=2682, shapes=4,
                        desc="cfg2 with per-env body shapes: 4 body shapes x 1024 envs interleaved in one batch (smplsim_create_shapes)"),
}
_WL = "cfg2"


def make_cfg(wl=None):
    from smplsim_b200.cfg import make_cfg as mk
    w = WORKLOADS[wl or _WL]
    return mk(env=w["env"], robot=w["robot"], overrides=w["overrides"])


DUMP_BYTES = 64 * 10 ** 6           # --dump-outputs: at most this much in all
PEAK_FP32_TFLOPS = 148 * 128 * 2 * 1.965e9 / 1e12     # 148 SMs x 128 FP32 lanes x 2 (FMA) x clocks.max.sm: 74.5 TFLOP/s nominal


def kernel_counters():
    """ncu counters of the dominant kernel (profiles/k_step5_counters.json, written from the committed ncu capture):
    issue-slot utilisation, active threads per instruction, resident warps, FP32 operations per env-step."""
    p = os.path.join(ROOT, "profiles", "k_step5_counters.json")
    try:
        return json.load(open(p))
    except Exception:
        return None


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region (B200_PROFILING.md recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.lines = []
        self.proc = None
        self.gpu = gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": float(max(mx)) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def dump_outputs(path, outs):
    """Write each array of `outs` ([envs, ...], float32) as path/<name>.npy.  Above DUMP_BYTES in all, a fixed seeded sample of the
    envs is written instead, with their indices in env_ids.npy."""
    os.makedirs(path, exist_ok=True)
    n = len(next(iter(outs.values())))
    row = sum(a[0].nbytes for a in outs.values()) + 8
    if n * row > DUMP_BYTES:
        ids = np.sort(np.random.default_rng(0).choice(n, DUMP_BYTES // row, replace=False))
        outs = {k: a[ids] for k, a in outs.items()}
        outs["env_ids"] = ids.astype(np.float64)
    for k, a in outs.items():
        np.save(os.path.join(path, f"{k}.npy"), a)


def measured_peak_hbm():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured"
        except Exception:
            pass
    return 6650.0, "fallback"


def host_cores():
    """Host threads this process can really run at once: CPU affinity, capped by the cgroup CPU quota (a container that sees
    128 logical CPUs is often limited to far fewer by cpu.max)."""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            txt = open(path).read().split()
            if path.endswith("cpu.max"):
                if txt[0] != "max":
                    n = min(n, max(1, int(np.ceil(int(txt[0]) / int(txt[1])))))
            else:
                q = int(txt[0])
                if q > 0:
                    per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
                    n = min(n, max(1, int(np.ceil(q / per))))
            break
        except Exception:
            continue
    return n


class CpuOracle:
    """The fp64 oracle port stepping a bounded sample of the cfg2 workload on `threads` host threads."""

    def __init__(self, threads=None):
        from oracle import oracle as orc
        self.orc = orc
        self.om = orc.OracleModel.from_cfg(make_cfg(), seed=0)
        self.logical = os.cpu_count() or 1
        self.rng = np.random.default_rng(0)
        self.per_step = None
        if threads is None:          # fixed rule, no calibration: one pthread per host core this process may use (affinity / cgroup quota)
            threads = host_cores()
        self._setup(threads)

    def _setup(self, threads):
        self.cores = threads
        self.nenv = 2 * self.cores
        self.envs = [self.orc.OracleEnv(self.om, env_id=i) for i in range(self.nenv)]
        for e in self.envs:
            e.reset()
        self.per_step = None

    def run(self, nsteps):
        a = np.clip(self.rng.normal(size=(nsteps, self.nenv, self.om.model.nu)) * SIGMA, -1, 1)
        t0 = time.perf_counter()
        self.orc.bench_env_steps(self.om, self.envs, a, autoreset=True, nthreads=self.cores)
        return time.perf_counter() - t0

    def sample(self, seconds_target):
        if self.per_step is None:
            self.run(2)                                   # thread start-up, page-in
            self.per_step = max(self.run(8) / 8, 1e-4)    # calibration
        nsteps = int(max(2, min(4000, seconds_target / self.per_step)))
        t = self.run(nsteps)
        self.per_step = t / nsteps
        return dict(value=self.nenv * nsteps / t, unit="env-steps/s", cores=self.cores, per_core=self.nenv * nsteps / t / self.cores, kind="port",
                    sample=f"{self.nenv} envs x {nsteps} env-steps ({self.nenv * nsteps} env-steps, {t:.1f} s) of the cfg2 workload, "
                           f"fp64 oracle port, {self.cores} pthreads (affinity / cgroup quota; {self.logical} logical CPUs visible)")


def cpu_oracle_throughput(seconds_target=12.0, threads=None):
    return CpuOracle(threads).sample(seconds_target)


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    co = CpuOracle()
    per = []
    cb = None
    budget = 150.0 / max(1, args.steps + args.warmup)      # the whole run ends within a few minutes
    secs = max(0.25, min(20.0, budget))
    if os.environ.get("SMPLSIM_BENCH_SECS"):              # tests: shrink the bounded sample
        secs = float(os.environ["SMPLSIM_BENCH_SECS"])
    t_run = time.perf_counter()
    for i in range(args.warmup + args.steps):
        cb = co.sample(secs)
        if i >= args.warmup:
            per.append(cb["value"])
    val = float(np.mean(per))
    ms_per = (time.perf_counter() - t_run) * 1e3 / max(1, args.warmup + args.steps)
    cb["value"] = val
    cb["sample"] = f"{args.steps} samples, each: " + cb["sample"]
    line = {
        "impl": "reference", "metric": "env-steps/sec SMPL humanoid (speed task, 15 substeps/step)", "value": val, "unit": "env-steps/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": {"workload": WORKLOAD, "note": "CPU oracle port; each step = one bounded sample"},
        "cpu_baseline": cb, "e2e": {"value": val, "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def measure(wl, args, torch, dist, world, rank, local, K, W, headline):
    """One workload on this rank's GPU: device-resident throughput, kernel time, end-to-end with host buffers (headline only)."""
    from smplsim_b200.batched import HumanoidBatchB200
    dev = torch.device(f"cuda:{local}")
    spec = WORKLOADS[wl]
    N = args.envs_per_gpu if headline else spec["envs"]
    cfg = make_cfg(wl)
    kw = {}
    if spec.get("shapes"):   # synthetic body shapes (no SMPL files here), interleaved over the envs
        from smplsim_b200.abi import model_from_cfg
        from smplsim_b200 import model as M
        base, m0 = M.load_parsed("smpl"), model_from_cfg(cfg)
        S = int(spec["shapes"])
        var = [dict(), dict(leg=1.15, arm=0.9, trunk=1.05, girth=1.1, density=1.1), dict(leg=0.88, arm=1.08, trunk=0.95, girth=0.92, density=0.95),
               dict(leg=1.05, arm=1.05, trunk=1.1, girth=1.2, density=1.0)]
        e = cfg.env
        kw["models"] = [M.build_model(M.shape_variant(base, **var[k % len(var)]), timestep=m0.timestep, contact_bodies=list(e.contact_bodies),
                                      control_mode=e.control_mode, clip_actions=bool(e.clip_actions), power_scale=float(e.power_scale))
                        for k in range(S)]
        kw["env_model"] = (np.arange(N) % S).astype(np.int32)
    env = HumanoidBatchB200(cfg, num_envs=N, device=str(dev), seed=0, rank=rank, with_aux=False, **kw)
    nu = env.num_actions
    gen = torch.Generator(device=dev)
    gen.manual_seed(0 + rank)
    motion = bool(spec.get("motion"))
    lib = None
    if motion:
        from smplsim_b200.motion_lib import MotionLibB200, synthetic_tables
        lib = MotionLibB200(env, synthetic_tables(env, num_clips=64, frames=300))
        ids = (torch.arange(N, device=dev) % 64).to(torch.int32)
        t_env = torch.rand(N, generator=gen, device=dev) * 8.0
        dt = float(env.dt)

    def draw(k):
        return torch.clamp(torch.randn(k, N, nu, generator=gen, device=dev) * SIGMA, -1, 1)

    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)      # > 126 MB L2

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def one_step(a):
        if motion:   # reference-pose feed of the step (motion_lib_base.py:313-354), then the step, then MoCap reset of finished envs
            st = lib.get_motion_state_intervaled(ids, t_env)
            out = env.step(a)
            env.reset(env.reset_buf, init_mode=2, qpos0=st["qpos"], qvel0=st["qvel"])
            t_env.add_(dt)
            t_env.masked_fill_(t_env > 9.0, 0.0)
        else:
            out = env.step(a); env.reset_done()
        return out

    if motion:
        st0 = lib.get_motion_state_intervaled(ids, t_env)
        env.reset(None, init_mode=2, qpos0=st0["qpos"], qvel0=st0["qvel"])
    else:
        env.reset()
    acts = draw(W)
    for i in range(W):
        one_step(acts[i]); flush.zero_()
    # ---------------- timed region 1: device-resident inputs ("value")
    acts = draw(K)
    launches0 = env.gpu_launches
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sampler = ClockSampler(local)
    if rank == 0 and headline:
        sampler.start()
    barrier()
    ev0.record()
    for i in range(K):
        last = one_step(acts[i]); flush.zero_()
    ev1.record()
    barrier()
    ms = ev0.elapsed_time(ev1)
    # what the caller holds after the last timed step (obs after the in-stream reset of the envs that finished), before the
    # kernel timing below steps the env again
    outputs = {k: t.float().cpu().numpy() for k, t in zip(("obs", "reward", "terminated", "truncated"), last)} \
        if headline and args.dump_outputs else None
    launches = env.gpu_launches - launches0
    # ---------------- the L2 flush alone (it sits inside the timed region above: `value` is conservative by this much)
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    f0.record()
    for i in range(10):
        flush.zero_()
    f1.record()
    torch.cuda.synchronize()
    flush_ms = f0.elapsed_time(f1) / 10
    # ---------------- per-kernel timing of k_step for the roofline (events on the launching stream)
    kev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(min(K, 50))]
    for i, (a, b) in enumerate(kev):
        flush.zero_()
        a.record(); env.step(acts[i % K]); b.record()
        env.reset_done()
    torch.cuda.synchronize()
    k_ms = float(np.mean([a.elapsed_time(b) for a, b in kev]))
    e2e_ms, Ke = 0.0, 0
    if headline:
        # ---------------- timed region 2: end to end through the public API with HOST buffers ("e2e")
        h_act = [torch.clamp(torch.randn(N, nu) * SIGMA, -1, 1).pin_memory() for _ in range(4)]
        h_obs = torch.empty(N, env.num_obs).pin_memory()
        h_rew = torch.empty(N).pin_memory()
        h_term = torch.empty(N, dtype=torch.uint8).pin_memory()
        h_trunc = torch.empty(N, dtype=torch.uint8).pin_memory()
        Ke = min(K, 100)

        def e2e_step(i):
            a = h_act[i % 4].to(dev, non_blocking=True)
            obs, rew, term, trunc = env.step(a)
            h_obs.copy_(obs, non_blocking=True); h_rew.copy_(rew, non_blocking=True)
            h_term.copy_(term, non_blocking=True); h_trunc.copy_(trunc, non_blocking=True)
            env.reset_done()
            flush.zero_()
            torch.cuda.current_stream().synchronize()       # the caller owns the host results before the next step

        for i in range(3):
            e2e_step(i)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        e0.record()
        for i in range(Ke):
            e2e_step(i)
        e1.record()
        barrier()
        e2e_ms = max(e0.elapsed_time(e1), (time.perf_counter() - t0) * 1e3)
    clocks = sampler.stop() if (rank == 0 and headline) else None
    # ---------------- max over ranks
    t = torch.tensor([ms, e2e_ms, k_ms, flush_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms, e2e_ms, k_ms, flush_ms = [float(x) for x in t.tolist()]
    out = dict(N=N, K=K, ms=ms, e2e_ms=e2e_ms, Ke=Ke, k_ms=k_ms, flush_ms=flush_ms, launches=launches, clocks=clocks, env=env, cfg=cfg,
               outputs=outputs)
    return out


def measure_ppo(torch, dist, world, rank, local, horizon=12, iters=2):
    """The one collective of the project (SURVEY 8e): a PPO iteration = device-resident rollout of `horizon` steps over this
    rank's 4 096 envs (policy forward included) -> GAE -> AgentPPO.update_params (10 full-batch epochs, the reference's 6-layer
    2048...512 MLP) with the gradients averaged over ranks by bucketed asynchronous NCCL all-reduces.  Max over ranks."""
    from smplsim_b200.batched import HumanoidBatchB200
    from smplsim_b200.cfg import make_cfg as mk
    from smplsim_b200.dist import rank_seed
    from smplsim_b200.learning import BatchedSampler
    from smplsim_b200.ppo import PolicyGaussian, PPOLearner, Value
    dev = torch.device(f"cuda:{local}")
    N = 4096
    units = [2048, 1536, 1024, 1024, 512, 512]           # data/cfg/learning/simple_mlp.yaml
    torch.manual_seed(0)
    env = HumanoidBatchB200(mk(env="speed"), num_envs=N, device=str(dev), seed=0, rank=rank, with_aux=False)
    policy = PolicyGaussian(env.num_obs, env.num_actions, units, "silu", -2.5, True).to(dev)
    value = Value(env.num_obs, units, "silu").to(dev)
    learner = PPOLearner(policy, value)
    gen = torch.Generator(device=dev); gen.manual_seed(rank_seed(0, rank))

    def act(obs):
        policy.eval()
        return policy.select_action(obs, generator=gen)

    sampler = BatchedSampler(env, act)
    ts, tu = [], []
    for it in range(iters + 1):
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(); t0 = time.perf_counter()
        batch = sampler.sample(horizon)
        torch.cuda.synchronize(); t1 = time.perf_counter()
        learner.update(batch)
        torch.cuda.synchronize(); t2 = time.perf_counter()
        if it > 0:
            ts.append(t1 - t0); tu.append(t2 - t1)
    t = torch.tensor([float(np.mean(ts)), float(np.mean(tu))], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    s_s, u_s = [float(x) for x in t.tolist()]
    nparam = sum(p.numel() for p in policy.parameters()) + sum(p.numel() for p in value.parameters())
    return {"workload": f"PPO iteration: {horizon}-step rollout x {N} envs/GPU (policy forward on device) + GAE + 10 full-batch epochs, MLP {units}",
            "samples_per_iter": horizon * N * world, "sample_s": s_s, "update_s": u_s, "sample_env_steps_per_s": horizon * N * world / s_s,
            "iter_samples_per_s": horizon * N * world / (s_s + u_s), "grad_bytes_allreduced_per_epoch": 4 * nparam if world > 1 else 0,
            "collective": "NCCL all-reduce of policy+value gradients (per-layer buckets, async) and of the advantage / RunningNorm moments"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--envs-per-gpu", type=int, default=ENVS_PER_GPU)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--workload", default="cfg2", choices=sorted(WORKLOADS))
    ap.add_argument("--no-extra", action="store_true", help="skip the short cfg4 / cfg5 runs appended to the headline line")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step returned (obs, reward, terminated, truncated) "
                                                          "as DIR/<name>.npy in float32; same arguments, same inputs")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the b200 path")
    global _WL, WORKLOAD, B_ALG_BYTES
    _WL = args.workload
    WORKLOAD, B_ALG_BYTES = WORKLOADS[_WL]["desc"], WORKLOADS[_WL]["balg"]
    if args.envs_per_gpu == ENVS_PER_GPU:
        args.envs_per_gpu = WORKLOADS[_WL]["envs"]
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local}"))
    torch.cuda.set_device(local)
    K, W = args.steps, max(3, args.warmup)
    r = measure(_WL, args, torch, dist, world, rank, local, K, W, True)
    env, cfg, N = r["env"], r["cfg"], r["N"]
    extra = {}
    if not args.no_extra and _WL == "cfg2":
        # the configurations north_star states its target on (cfg4: 65 536 envs + motion feed on 8 GPUs; cfg5: SMPL-X), short runs
        for wl in ("cfg4", "cfg5", "cfg2-selfcol", "cfg2-shapes"):
            Kx = max(10, K // 8)
            x = measure(wl, args, torch, dist, world, rank, local, Kx, 3, False)
            extra[wl] = {"workload": WORKLOADS[wl]["desc"], "envs_per_gpu": x["N"], "global_envs": x["N"] * world, "steps": Kx,
                         "value": x["N"] * world * Kx / (x["ms"] * 1e-3), "unit": "env-steps/s", "ms_per_step": x["ms"] / Kx,
                         "kernel_ms": x["k_ms"], "gpu_launches": x["launches"], "smem_bytes_per_env": x["env"].smem_bytes_per_env()}
            del x
        extra["ppo"] = measure_ppo(torch, dist, world, rank, local)
    if rank == 0:
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, r["outputs"])
        ms, e2e_ms, k_ms, Ke = r["ms"], r["e2e_ms"], r["k_ms"], r["Ke"]
        nu = env.num_actions
        total_envs = N * world
        value = total_envs * K / (ms * 1e-3)
        e2e = total_envs * Ke / (e2e_ms * 1e-3)
        peak, peak_src = measured_peak_hbm()
        balg = B_ALG_BYTES + (B_ALG_STALE_BYTES if env.envcfg.spd_stale and env.envcfg.control_mode == 0 else 0)
        achieved = balg * N / (k_ms * 1e-3) / 1e9
        traffic = None
        kc = kernel_counters() if _WL == "cfg2" else None
        secondary = None
        if kc:
            traffic = kc.get("dram_bytes_per_launch")
            flops = kc.get("fp32_flops_per_env_step")
            secondary = {"issue_active_pct": kc.get("issue_active_pct"), "threads_per_inst": kc.get("threads_per_inst"),
                         "warps_per_sm": kc.get("warps_per_sm"), "warp_inst_per_env_step": kc.get("warp_inst_per_env_step"),
                         "fp32_flops_per_env_step": flops,
                         "fp32_tflops": (flops * N / (k_ms * 1e-3) / 1e12) if flops else None,
                         "fp32_flop_frac": (flops * N / (k_ms * 1e-3) / 1e12 / PEAK_FP32_TFLOPS) if flops else None,
                         "fp32_peak_tflops": PEAK_FP32_TFLOPS, "source": kc.get("source")}
        line = {
            "metric": "env-steps/sec SMPL humanoid (speed task, 15 substeps/step)", "value": value, "unit": "env-steps/s", "n_gpus": world,
            "steps": K, "warmup": W, "ms_per_step": ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic",
            "config": {"workload": WORKLOAD, "envs_per_gpu": N, "global_envs": total_envs, "substeps_per_step": int(env.envcfg.nsubsteps),
                       "control_mode": str(cfg.env.control_mode), "spd_inertia": "stale" if env.envcfg.spd_stale else "fresh", "parallelism": f"env-shard x{world}",
                       "kernel": f"v{env.kernel_version}", "smem_bytes_per_env": env.smem_bytes_per_env(),
                       "l2": "256 MiB flush buffer zeroed after every step inside the timed region (state ~11 MB < 126 MB L2)",
                       "flush_ms_per_step": r["flush_ms"], "value_excluding_flush": total_envs * K / (max(ms - K * r["flush_ms"], 1e-9) * 1e-3)},
            "substeps_per_s": value * int(env.envcfg.nsubsteps),
            "e2e": {"value": e2e, "unit": "env-steps/s", "h2d_bytes_per_step": N * nu * 4, "d2h_bytes_per_step": N * (env.num_obs * 4 + 4 + 2),
                    "steps": Ke, "note": "pinned host actions -> device, step, obs/reward/flags -> pinned host, stream sync every step"},
            "gpu_launches": r["launches"], "clocks": r["clocks"],
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                         "peak_source": peak_src, "kernel": f"k_step{env.kernel_version}", "kernel_ms": k_ms, "alg_bytes_per_env_step": balg,
                         "secondary": secondary,
                         "note": "15 fused substeps keep state on-chip: the kernel is FP32-issue / latency bound, not HBM bound (SURVEY.md 8d); "
                                 "`secondary` carries the issue-slot and FP32 fractions"},
        }
        if extra:
            line["other_workloads"] = extra
        if not args.no_cpu_baseline and world == 1:
            line["cpu_baseline"] = cpu_oracle_throughput()
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
