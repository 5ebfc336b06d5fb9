#!/usr/bin/env python
"""Generate tests/golden/*.npz by running the REFERENCE's own numpy code.

Run in the build container only (needs /root/reference; it does not exist on the GPU box):

    python tests/golden/make_golden.py

The reference cannot be imported as-is here (mujoco, gymnasium, lxml, ... are absent;
SURVEY.md 8c), so the absent third-party modules are replaced by stubs *before* importing
smpl_sim.envs.*; every function exercised below is pure numpy/scipy and runs unmodified:

  compute_humanoid_self_obs_v1/_v2      smpl_sim/envs/humanoid_env.py:565-688
  compute_speed_observations/forward_reward   smpl_sim/envs/tasks/humanoid_speed.py:9-46
  compute_location_observations/reach_reward  smpl_sim/envs/tasks/humanoid_reach.py:10-30
  height_reward                         smpl_sim/envs/tasks/humanoid_getup.py:9-18
  StablePDController / PIDController / SimpleTorqueController.control  smpl_sim/envs/controllers.py
  HumanoidEnv.build_pd_action_scale     smpl_sim/envs/humanoid_env.py:325-370
  MotionLibBase._calc_frame_blend       smpl_sim/smpllib/motion_lib_base.py:448-458

Inputs are seeded; the mass matrices fed to the stable-PD controller come from
smplsim_b200.model.mass_matrix_numpy (plain Jacobian sum, independent of oracle and CUDA).
"""
import os
import sys
import types
from unittest.mock import MagicMock

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.abspath(os.path.join(HERE, "..", ".."))
REF = os.environ.get("SMPLSIM_REFERENCE", "/root/reference")
sys.path.insert(0, REPO)
sys.path.insert(0, REF)

# ---- stubs for absent third-party modules
gym = types.ModuleType("gymnasium")


class _Env:
    def reset(self, seed=None, options=None):
        pass


gym.Env = _Env
gym.spaces = MagicMock()
sys.modules["gymnasium"] = gym
import importlib.abc  # noqa: E402
import importlib.machinery  # noqa: E402


class _StubFinder(importlib.abc.MetaPathFinder, importlib.abc.Loader):
    """Last-resort finder: any third-party module that is absent from this image becomes a MagicMock."""

    def find_spec(self, fullname, path, target=None):
        if fullname.split(".")[0] not in _STUBBED:
            return None
        return importlib.machinery.ModuleSpec(fullname, self, is_package=True)

    def create_module(self, spec):
        mod = MagicMock(name=spec.name)
        mod.__path__ = []
        mod.__spec__ = spec
        return mod

    def exec_module(self, module):
        pass


_STUBBED = {"mujoco"}
sys.meta_path.append(_StubFinder())


def _import_with_stubs(fn):
    """Call fn(); every time a third-party module is missing, stub its top-level name and retry."""
    for _ in range(64):
        try:
            return fn()
        except ModuleNotFoundError as e:
            top = e.name.split(".")[0]
            if top in ("smpl_sim", "smplsim_b200") or top in _STUBBED:
                raise
            _STUBBED.add(top)
            for k in [k for k in sys.modules if k.startswith("smpl_sim")]:
                if not isinstance(sys.modules[k], MagicMock):
                    del sys.modules[k]
    raise RuntimeError("too many missing modules")


# modules of the reference itself that only matter for model building / legacy envs
for name in ["smpl_sim.smpllib.smpl_local_robot", "smpl_sim.smpllib.smpl_xml_addons", "smpl_sim.smpllib.motion_lib_base",
             "smpl_sim.envs.smplenv", "smpl_sim.smpllib.smpl_mujoco_new"]:
    sys.modules[name] = MagicMock()
import mujoco  # noqa: E402  (the stub)



def _load_reference():
    from smpl_sim.envs import humanoid_env as HE
    from smpl_sim.envs import controllers as CT
    from smpl_sim.envs.tasks import humanoid_speed as HS
    from smpl_sim.envs.tasks import humanoid_reach as HR
    from smpl_sim.envs.tasks import humanoid_getup as HG
    return HE, CT, HS, HR, HG


HE, CT, HS, HR, HG = _import_with_stubs(_load_reference)
print("stubbed third-party modules:", sorted(_STUBBED))

from smplsim_b200.model import load_model, mass_matrix_numpy, fk_numpy  # noqa: E402


def rand_quat(rng, n):
    q = rng.normal(size=(n, 4))
    return q / np.linalg.norm(q, axis=-1, keepdims=True)


def gen_obs(model_name, nb, nu, seed, B=48):
    rng = np.random.default_rng(seed)
    m = load_model(model_name)
    assert m.nbody == nb
    qpos = np.zeros((B, m.nq))
    qpos[:, 0:2] = rng.uniform(-20, 20, (B, 2))
    qpos[:, 2] = rng.uniform(0.2, 1.2, B)
    qpos[:, 3:7] = rand_quat(rng, B)
    qpos[:, 7:] = rng.uniform(-1.2, 1.2, (B, nu))
    qpos[0, 3:7] = [0.5, 0.5, 0.5, 0.5]                    # K-7a: Default pose
    qpos[0, 7:] = 0
    qpos[0, 0:3] = [0, 0, 0.94]
    qvel = rng.normal(size=(B, m.nv)) * 2
    xpos = np.zeros((B, nb, 3))
    xquat = np.zeros((B, nb, 4))
    for i in range(B):
        xpos[i], xquat[i], _ = fk_numpy(m, qpos[i])
    linvel = rng.normal(size=(B, nb, 3))
    angvel = rng.normal(size=(B, nb, 3)) * 3
    out = dict(qpos=qpos, qvel=qvel, xpos=xpos, xquat=xquat, linvel=linvel, angvel=angvel)
    for upright in (False, True):
        for rh in (True, False):
            if upright and not rh:          # read by no test; with it obs_smpl.npz would pass 1 MB
                continue
            tag = f"u{int(upright)}h{int(rh)}"
            # the reference's remove_base_rot only works for batch size 1 (np.repeat semantics,
            # np_transform_utils.py:145-146), which is how the env calls it ([None,] at humanoid_env.py:391-394)
            v1, v2 = [], []
            for i in range(B):
                s = slice(i, i + 1)
                d1 = HE.compute_humanoid_self_obs_v1(qpos[s], qvel[s], xpos[s], xquat[s], upright, rh, model_name)
                d2 = HE.compute_humanoid_self_obs_v2(xpos[s], xquat[s], linvel[s], angvel[s], upright, rh, model_name)
                v1.append(np.concatenate([v.ravel() for v in d1.values()]))
                v2.append(np.concatenate([v.ravel() for v in d2.values()]))
            out["v1_" + tag] = np.array(v1)
            out["v2_" + tag] = np.array(v2)
    # task obs / rewards (single-env functions in the reference)
    tar_speed = rng.uniform(0, 5, B)
    tar_pos = rng.uniform(-1, 2, (B, 3))
    prev_root = xpos[:, 0] - rng.normal(size=(B, 3)) * 0.05
    sp_obs, rc_obs, sp_rew, rc_rew, gu_rew = [], [], [], [], []
    tar_h = rng.uniform(0.5, 1.2, B)
    for i in range(B):
        d = HS.compute_speed_observations(qpos[i:i + 1, 3:7], tar_speed[i], False, model_name)
        sp_obs.append(np.concatenate([v.ravel() for v in d.values()]))
        d = HR.compute_location_observations(qpos[i:i + 1, 0:3], qpos[i:i + 1, 3:7], tar_pos[i:i + 1], False, model_name)
        rc_obs.append(np.concatenate([v.ravel() for v in d.values()]))
        sp_rew.append(HS.forward_reward(tar_speed[i], xpos[i:i + 1, 0], prev_root[i:i + 1], 1 / 30.0)[0])
        rc_rew.append(HR.reach_reward(xpos[i:i + 1, -1], tar_pos[i:i + 1])[0])
        gu_rew.append(HG.height_reward(np.array([[tar_h[i]]]), xpos[i:i + 1, 0])[0])
    out.update(tar_speed=tar_speed, tar_pos=tar_pos, prev_root=prev_root, tar_h=tar_h, speed_obs=np.array(sp_obs),
               reach_obs=np.array(rc_obs), speed_rew=np.array(sp_rew), reach_rew=np.array(rc_rew), getup_rew=np.array(gu_rew))
    np.savez_compressed(os.path.join(HERE, f"obs_{model_name}.npz"), **out)
    print(f"obs_{model_name}.npz: v1 {out['v1_u0h1'].shape} v2 {out['v2_u0h1'].shape}; "
          f"K-7a sum v2 = {out['v2_u0h1'][0].sum() - out['v2_u0h1'][0][-6 * nb:].sum():.4f}")


def gen_controllers(seed=7, B=12):
    rng = np.random.default_rng(seed)
    m = load_model("smpl")
    nv, nu = m.nv, m.nu

    # --- gains / action scale through the reference's own build_pd_action_scale
    class FakeJoint:
        def __init__(self, r):
            self.range = r

    class FakeModel:
        def joint(self, n):
            return FakeJoint(m.dof_range[6 + m.joint_names.index(n)])

    gains = {}
    for mode in ("uhc_pd", "pd"):
        fake = types.SimpleNamespace(dof_size=nu, actuator_names=list(m.joint_names), mj_model=FakeModel(), control_mode=mode,
                                     clip_actions=True)
        HE.HumanoidEnv.build_pd_action_scale(fake)
        gains[mode] = fake
    f = gains["uhc_pd"]
    out = dict(jkp=f.jkp, jkd=f.jkd, torque_lim=f.torque_lim, pd_action_scale=f._pd_action_scale, pd_action_offset=f._pd_action_offset)

    # --- controllers: mujoco.mj_fullM shim expands "qM" (we pass the dense matrix through)
    def mj_fullM(model, dst, qM):
        dst[:] = np.asarray(qM).reshape(dst.shape)

    mujoco.mj_fullM = mj_fullM
    spd = CT.StablePDController(f._pd_action_scale, f._pd_action_offset, nv, f.torque_lim, f.jkp, f.jkd)
    pid = CT.PIDController(f._pd_action_scale, f._pd_action_offset, f.torque_lim, f.jkp, f.jkd, np.zeros_like(f.jkd))
    trq = CT.SimpleTorqueController(10.0 * f.torque_lim, f.torque_lim)
    qpos = np.zeros((B, m.nq))
    qpos[:, 2] = 0.9
    qpos[:, 3:7] = rand_quat(rng, B)
    qpos[:, 7:] = rng.uniform(-1.0, 1.0, (B, nu))
    qvel = rng.normal(size=(B, nv))
    qpos_stale = qpos.copy()
    qpos_stale[:, 7:] += rng.normal(size=(B, nu)) * 0.01        # M is evaluated at a slightly older state (quirk Q1)
    action = np.clip(rng.normal(size=(B, nu)) * 0.5, -1, 1)
    Cbias = rng.normal(size=(B, nv)) * 20
    Ms = np.zeros((B, nv, nv))
    t_spd, t_pid, t_trq = [], [], []
    for i in range(B):
        Ms[i], _ = mass_matrix_numpy(m, qpos_stale[i])
        mj_model = types.SimpleNamespace(opt=types.SimpleNamespace(timestep=1.0 / 450.0), nv=nv)
        mj_data = types.SimpleNamespace(qpos=qpos[i].copy(), qvel=qvel[i].copy(), qM=Ms[i].copy(), qfrc_bias=Cbias[i].copy())
        t_spd.append(spd.control(action[i], mj_model, mj_data))
        mj_data = types.SimpleNamespace(qpos=qpos[i].copy(), qvel=qvel[i].copy())
        t_pid.append(pid.control(action[i], mj_model, mj_data))
        t_trq.append(trq.control(action[i], mj_model, mj_data))
    out.update(qpos=qpos, qvel=qvel, qpos_stale=qpos_stale, action=action, C=Cbias, M=Ms, torque_spd=np.array(t_spd),
               torque_pd=np.array(t_pid), torque_torque=np.array(t_trq))
    np.savez_compressed(os.path.join(HERE, "controllers_smpl.npz"), **out)
    print("controllers_smpl.npz: |tau_spd| max", np.abs(out["torque_spd"]).max(), "clipped frac",
          float(np.mean(np.abs(out["torque_spd"]) >= f.torque_lim[None] - 1e-9)))


def gen_simple_pid(seed=11, T=40):
    """SimplePID (controllers.py:186-262) as humanoid_env.setup_controller builds it (:318-319): Kp = jkp/10, Ki = 1, Kd = jkd/10,
    dt = timestep * control_freq_inv, stateful (integral, last error) across calls -- a T-call sequence on one controller."""
    rng = np.random.default_rng(seed)
    m = load_model("smpl")
    nu = m.nu

    class FakeJoint:
        def __init__(self, r):
            self.range = r

    class FakeModel:
        def joint(self, n):
            return FakeJoint(m.dof_range[6 + m.joint_names.index(n)])

    fake = types.SimpleNamespace(dof_size=nu, actuator_names=list(m.joint_names), mj_model=FakeModel(), control_mode="simple_pid", clip_actions=True)
    HE.HumanoidEnv.build_pd_action_scale(fake)
    dt = (1.0 / 450.0) * 15
    ctl = CT.SimplePID(fake.jkp / 10, np.ones_like(fake.jkp), fake.jkd / 10, dt, fake.torque_lim, fake._pd_action_scale, fake._pd_action_offset)
    q = rng.uniform(-0.5, 0.5, nu)
    qs, acts, taus = [], [], []
    for t in range(T):
        if t % 5 == 0:
            a = np.clip(rng.normal(size=nu) * 0.3, -1, 1)
        q = q + rng.normal(size=nu) * 0.01
        qpos = np.zeros(m.nq); qpos[7:] = q
        tau = ctl.control(a, None, types.SimpleNamespace(qpos=qpos))
        qs.append(qpos.copy()); acts.append(a.copy()); taus.append(np.array(tau).copy())
    np.savez_compressed(os.path.join(HERE, "simple_pid_smpl.npz"), qpos=np.array(qs), action=np.array(acts), torque=np.array(taus), dt=dt,
                        jkp=fake.jkp, jkd=fake.jkd, torque_lim=fake.torque_lim)
    print("simple_pid_smpl.npz: |tau| max", np.abs(np.array(taus)).max(), "clipped frac", float(np.mean(np.abs(np.array(taus)) >= fake.torque_lim[None] - 1e-9)))


def gen_frame_blend(seed=3, B=256):
    """MotionLibBase._calc_frame_blend + the frame index expression of get_motion_state_intervaled
    (motion_lib_base.py:321-323,448-458) -- executed from the reference source text, since importing the
    module needs joblib/smplx/torch-geometry stubs that would replace the function under test."""
    import ast
    import inspect  # noqa: F401
    src = open(os.path.join(REF, "smpl_sim/smpllib/motion_lib_base.py")).read()
    tree = ast.parse(src)
    fn = None
    for node in ast.walk(tree):
        if isinstance(node, ast.FunctionDef) and node.name == "_calc_frame_blend":
            fn = node
    mod = ast.Module(body=[fn], type_ignores=[])
    ns = {"np": np}
    exec(compile(mod, "motion_lib_base.py", "exec"), ns)
    calc = ns["_calc_frame_blend"]
    rng = np.random.default_rng(seed)
    num_frames = rng.integers(2, 400, B)
    dt = np.full(B, 1.0 / 30.0)
    mlen = dt * (num_frames - 1)
    t = rng.uniform(-0.5, 1.3, B) * mlen
    t[:8] = [0.0, -1.0, mlen[2], mlen[3] * 2, dt[4] * 3, dt[5] * 3 - 1e-9, dt[6] * 3 + 1e-9, 0.5 * dt[7]]
    i0, i1, blend = calc(None, t, mlen, num_frames, dt)
    frame_idx = ((1.0 - blend) * i0 + blend * i1).astype(int)
    np.savez_compressed(os.path.join(HERE, "frame_blend.npz"), time=t, motion_len=mlen, num_frames=num_frames, dt=dt, frame_idx=frame_idx)
    print("frame_blend.npz:", frame_idx[:8])


def gen_gae(seed=5, T=24, N=6):
    """estimate_advantages (smpl_sim/learning/learning_utils.py:198-218) on N concatenated env columns of length T; every column
    ends with not_done = 0 (as every sampled trajectory does in Agent.sample_worker), so the flat recursion restarts per column."""
    import torch
    LU = _import_with_stubs(lambda: __import__("smpl_sim.learning.learning_utils", fromlist=["x"]))
    rng = np.random.default_rng(seed)
    rew = rng.uniform(0, 1, (T, N)).astype(np.float32)
    val = rng.normal(size=(T, N)).astype(np.float32)
    not_dead = (rng.random((T, N)) > 0.06).astype(np.float32)
    not_done = not_dead * (rng.random((T, N)) > 0.05).astype(np.float32)
    not_done[-1] = 0
    flat = lambda a: torch.from_numpy(np.ascontiguousarray(a.T).reshape(-1, 1).copy())       # env-major concatenation
    adv, ret = LU.estimate_advantages(flat(rew), flat(not_done), flat(not_dead), flat(val), 0.99, 0.95)
    np.savez_compressed(os.path.join(HERE, "gae.npz"), rewards=rew, values=val, not_dead=not_dead, not_done=not_done,
                        advantages=adv.numpy().reshape(N, T).T, returns=ret.numpy().reshape(N, T).T)
    print("gae.npz:", adv.shape, float(adv.mean()), float(adv.std()))


if __name__ == "__main__":
    gen_gae()
    gen_obs("smpl", 24, 69, seed=11)
    gen_obs("smplx", 52, 153, seed=12, B=8)
    gen_controllers()
    gen_simple_pid()
    gen_frame_blend()
