"""GPU parity tests, part 2 (round 2): the holes the round-1 review listed.

  * the FUSED Humanoid step (physics on) against oracle physics + the numpy restatement of the reference's obs/reward;
  * the fused AnymalTerrain physics kernel (PD decimation loop, anymal_terrain.py:441-451, + the extra simulate of
    VecTask.step) against the oracle driven with the same PD law;
  * every task once at its BASELINE.json size and once at an N that is not a multiple of the envs-per-block
    (non-tile kernels, tail lanes);
  * B2G_FAST_TRIG=1 (the product build, __sincosf) against a B2G_FAST_TRIG=0 build of the same library;
  * the quad (specialised Ant) path against the generic Stepper path on identical inputs.
Tolerances as in tests/test_gpu_parity.py (fp32 engine vs fp64 oracle from identical states)."""
import copy
import os
import subprocess
import sys
import numpy as np
import pytest
import torch

from isaacgymenvs_b200.assets import load_compiled

pytestmark = pytest.mark.gpu
G = (0.0, 0.0, -9.81)
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
f32 = np.float32


def _make(task, n, **env_over):
    import isaacgymenvs_b200
    from isaacgymenvs_b200 import config
    cfg = config.builtin_cfg(task, {"sim_device": "cuda:0", "rl_device": "cuda:0"})
    cfg["task"]["env"].update(env_over)
    return isaacgymenvs_b200.make(seed=42, task=task, num_envs=n, sim_device="cuda:0", rl_device="cuda:0",
                                  headless=True, cfg=cfg)


def _loco_check(env, orc, task, steps, rng, full_obs=True):
    """steps of env.step() against oracle physics (+ numpy obs/reward when full_obs)."""
    from oracle import tasks_np as T
    n, nd = env.num_envs, env.num_dof
    hum = task == "Humanoid"
    lo, hi = env.dof_limits_lower_np, env.dof_limits_upper_np
    gears = env.motor_efforts_np.astype(f32)
    e = env.cfg["env"]
    dt = f32(env.cfg["sim"]["dt"])
    targets = np.tile(f32([1000, 0, 0]), (n, 1)); isr = np.tile(f32([0, 0, 0, 1]), (n, 1))
    b0 = np.tile(f32([1, 0, 0]), (n, 1)); b1 = np.tile(f32([0, 0, 1]), (n, 1))
    worst = dict(pos=0.0, q=0.0)
    for k in range(steps):
        r64 = env.root_states.cpu().numpy().astype(np.float64)
        d64 = env.dof_state.cpu().numpy().astype(np.float64).reshape(n, nd, 2)
        pot_in = env.potentials.cpu().numpy().copy()
        prog_in = env.progress_buf.cpu().numpy().copy()
        a = rng.uniform(-1.5, 1.5, size=(n, nd)).astype(f32)
        ac = np.clip(a, -1, 1)
        out = orc.simulate(r64, d64, (ac * gears[None] * f32(e["powerScale"])).astype(np.float64))
        obs, rew, reset, _ = env.step(torch.tensor(a, device=env.device))
        torch.cuda.synchronize()
        rg = env.root_states.cpu().numpy(); qg = env.dof_pos.cpu().numpy(); vg = env.dof_vel.cpu().numpy()
        sg = env.vec_sensor_tensor.cpu().numpy()
        keep = reset.cpu().numpy() == 0          # envs that terminate are re-initialised by the NEXT step, so all are comparable
        assert np.isfinite(rg).all() and np.isfinite(qg).all()
        if full_obs:
            if hum:
                fg = env.dof_force_tensor.cpu().numpy()
                o_np, pot, prev, _, _ = T.humanoid_observations(rg, targets, pot_in, isr, qg, vg, fg, lo, hi, e["dofVelocityScale"], sg, ac, dt,
                                                                e["contactForceScale"], e.get("angularVelocityScale", 0.1), b0, b1)
            else:
                o_np, pot, prev, _, _ = T.ant_observations(rg, targets, pot_in, isr, qg, vg, lo, hi, e["dofVelocityScale"], sg, ac, dt,
                                                           e["contactForceScale"], b0, b1)
            og = obs["obs"].cpu().numpy()
            d = np.abs(og - o_np)
            for col in (7, 8, 9):
                d[:, col] = np.minimum(d[:, col], np.abs(2 * np.pi - d[:, col]))
            assert (d / np.maximum(1, np.abs(o_np))).max() < 2e-6
            assert np.array_equal(env.potentials.cpu().numpy(), pot)
            if hum:
                r_np, reset_np = T.humanoid_reward(og, np.zeros(n, np.int64), prog_in + 1, ac, e["upWeight"], e["headingWeight"], pot, prev,
                                                   e["actionsCost"], e["energyCost"], e["jointsAtLimitCost"], float(gears.max()), gears,
                                                   e["terminationHeight"], e["deathCost"], float(e["episodeLength"]))
            else:
                r_np, reset_np = T.ant_reward(og, np.zeros(n, np.int64), prog_in + 1, ac, e["upWeight"], e["headingWeight"], pot, prev,
                                              e["actionsCost"], e["energyCost"], e["jointsAtLimitCost"], e["terminationHeight"], e["deathCost"],
                                              float(e["episodeLength"]))
            assert np.array_equal(reset.cpu().numpy(), reset_np)
            assert (np.abs(rew.cpu().numpy() - r_np) / np.maximum(1, np.abs(r_np))).max() < 1e-5
        # physics against the fp64 oracle (identical start states, one control step)
        worst["pos"] = max(worst["pos"], np.abs(rg[:, :7] - r64[:, :7]).max())
        worst["q"] = max(worst["q"], np.abs(qg - d64[..., 0]).max())
        assert np.abs(rg[:, :7] - r64[:, :7]).max() < 5e-5, (k, np.abs(rg[:, :7] - r64[:, :7]).max())
        dq = np.abs(qg - d64[..., 0])
        # Humanoid: joints driven against their stiff limit springs (k up to 6750 N m/rad, 200 N m motors) amplify fp32
        # round-off in a handful of DOFs; the bulk agrees to 2e-5, the worst case stays below 3e-4
        assert np.quantile(dq, 0.999) < (3e-5 if hum else 2e-5), np.quantile(dq, 0.999)
        assert dq.max() < (3e-4 if hum else 5e-5), dq.max()
        verr = np.abs(rg[:, 7:] - r64[:, 7:]) / np.maximum(1.0, np.abs(r64[:, 7:]))
        assert verr.max() < 2e-3
        ns = out["sensor"].shape[1]
        assert np.abs(sg.reshape(n, ns, 6) - out["sensor"]).max() < 5e-3 * max(1.0, np.abs(out["sensor"]).max())
        if hum:
            fg = env.dof_force_tensor.cpu().numpy()
            assert np.abs(fg - out["dof_force"]).max() < 5e-3 * max(1.0, np.abs(out["dof_force"]).max())
        if not keep.all():
            break
    return worst


def _loco_orc(env, threads=8):
    from oracle.oracle import OracleSim
    return OracleSim(env.model, env.cfg["sim"]["dt"], env.cfg["sim"]["substeps"], G, ground_mu=env.cfg["env"]["plane"]["dynamicFriction"], threads=threads)


def test_fused_humanoid_step_equals_oracle_pipeline():
    """loco_step_kernel<4,0,HUM=1,...> with physics on (the kernel the Humanoid bench times): first step resets every env,
    the following steps must equal oracle physics + the numpy restatement of compute_humanoid_observations / _reward
    (humanoid.py:323-413), including the staged dof_force tile."""
    n = 256
    env = _make("Humanoid", n)
    rng = np.random.default_rng(0)
    env.step(torch.tensor(rng.uniform(-1, 1, size=(n, 21)).astype(f32), device=env.device))      # resets every env
    torch.cuda.synchronize()
    assert (env.progress_buf == 0).all() and (env.reset_count == 1).all()
    q = env.dof_pos.cpu().numpy()
    assert (q >= env.dof_limits_lower_np - 1e-6).all() and (q <= env.dof_limits_upper_np + 1e-6).all()
    _loco_check(env, _loco_orc(env), "Humanoid", 5, rng)


@pytest.mark.parametrize("task,n", [("Ant", 16384), ("Humanoid", 8192), ("Ant", 1000), ("Ant", 1008), ("Humanoid", 1001), ("Ant", 17)])
def test_loco_baseline_sizes_and_tail_lanes(task, n):
    """BASELINE.json sizes (Ant 16384, Humanoid 8192) and sizes that are not whole tiles: N=1000 / 1001 / 17 run the
    non-tile kernels with invalid tail lanes, N=1008 is a multiple of 16 envs but not of 32."""
    env = _make(task, n)
    rng = np.random.default_rng(n)
    nd = env.num_dof
    env.step(torch.tensor(rng.uniform(-1, 1, size=(n, nd)).astype(f32), device=env.device))
    torch.cuda.synchronize()
    _loco_check(env, _loco_orc(env, threads=16), task, 3, rng)


def test_quad_path_equals_generic_path(tmp_path):
    """The specialised Ant step (b2g_quad.cuh) and the generic slot-program Stepper are two formulations of one
    sub-step: from identical states and actions, a whole control step agrees to fp32 round-off."""
    code = r'''
import os, sys, numpy as np, torch
sys.path.insert(0, %r)
import isaacgymenvs_b200
from isaacgymenvs_b200 import config
n = 512
cfg = config.builtin_cfg("Ant", {"sim_device": "cuda:0", "rl_device": "cuda:0"})
env = isaacgymenvs_b200.make(seed=42, task="Ant", num_envs=n, sim_device="cuda:0", rl_device="cuda:0", headless=True, cfg=cfg)
g = torch.Generator(device="cuda:0").manual_seed(5)
outs = []
for k in range(12):
    obs, rew, reset, _ = env.step(2 * torch.rand((n, 8), device="cuda:0", generator=g) - 1)
torch.cuda.synchronize()
np.savez(sys.argv[1], obs=obs["obs"].cpu().numpy(), rew=rew.cpu().numpy(), reset=reset.cpu().numpy(), root=env.root_states.cpu().numpy(),
         dof=env.dof_state.cpu().numpy(), sens=env.vec_sensor_tensor.cpu().numpy(), quad=np.int32(env.sim.quad_ns()))
''' % ROOT
    res = []
    for noquad in ("0", "1"):
        out = str(tmp_path / f"quadcmp_{noquad}.npz")
        env_ = dict(os.environ, B2G_NO_QUAD=noquad)
        subprocess.check_call([sys.executable, "-c", code, out], env=env_, cwd=ROOT)
        res.append(dict(np.load(out)))
    assert int(res[0]["quad"]) == 2 and int(res[1]["quad"]) == 0
    assert np.array_equal(res[0]["reset"], res[1]["reset"])
    rel = lambda a, b: (np.abs(a - b) / np.maximum(1.0, np.abs(b))).max()
    assert rel(res[0]["root"], res[1]["root"]) < 2e-3, rel(res[0]["root"], res[1]["root"])      # 12 contact-rich steps of round-off
    assert rel(res[0]["dof"], res[1]["dof"]) < 5e-3
    assert np.median(np.abs(res[0]["root"][:, :3] - res[1]["root"][:, :3]).max(1)) < 2e-5
    assert np.median(np.abs(res[0]["obs"] - res[1]["obs"]).max(1)) < 5e-4


# ------------------------------------------------------------------------------------ AnymalTerrain
def _make_anymal(n, terrain=None, **over):
    import isaacgymenvs_b200
    from isaacgymenvs_b200 import config
    cfg = config.builtin_cfg("AnymalTerrain", {"sim_device": "cuda:0", "rl_device": "cuda:0"})
    e = cfg["task"]["env"]
    if terrain:
        e["terrain"].update(terrain)
    for k, v in over.items():
        if k in e["learn"]:
            e["learn"][k] = v
        elif k in e["control"]:
            e["control"][k] = v
        else:
            e[k] = v
    return isaacgymenvs_b200.make(seed=42, task="AnymalTerrain", num_envs=n, sim_device="cuda:0", rl_device="cuda:0",
                                  headless=True, cfg=cfg)


def _anymal_check(env, steps, rng):
    """env.step() against the oracle driven by the same PD loop: decimation x {torque = clip(Kp (s a + q0 - q) - Kd qd),
    simulate} (anymal_terrain.py:441-451) then control_freq_inv x simulate with the last torques (vec_task.py:379-382)."""
    from oracle.oracle import OracleSim
    n, nd = env.num_envs, env.num_dof
    m = env.model
    sim_cfg = env.cfg["sim"]
    kw = {}
    if env.custom_origins:
        t = env.terrain
        kw = dict(hfield=np.asarray(t.heightsamples, np.float64).reshape(t.tot_rows, t.tot_cols) * t.vertical_scale, hf_scale=t.horizontal_scale,
                  hf_origin=(-t.border_size, -t.border_size))
    mu_g = env.cfg["env"]["terrain"]["dynamicFriction"]
    orc = OracleSim(m, sim_cfg["dt"], sim_cfg["substeps"], G, ground_mu=mu_g, threads=16, **kw)
    env.env_friction[:] = float(np.asarray(m.cp_mu)[0])       # one friction bucket: the oracle has one friction per sphere
    q0 = env.default_dof_pos[0].cpu().numpy().astype(np.float64)
    Kp, Kd, sc = float(env.Kp), float(env.Kd), float(env.action_scale)
    clip = float(env.clip_actions)
    cfi = int(env.control_freq_inv)
    n_cmp = 0
    for k in range(steps):
        r64 = env.root_states.cpu().numpy().astype(np.float64)
        d64 = env.dof_state.cpu().numpy().astype(np.float64).reshape(n, nd, 2)
        a = rng.uniform(-1, 1, size=(n, nd)).astype(f32)
        ac = np.clip(a, -clip, clip).astype(np.float64)
        tau = None
        for _ in range(env.decimation):
            tau = np.clip(Kp * (sc * ac + q0[None] - d64[..., 0]) - Kd * d64[..., 1], -80.0, 80.0)
            out = orc.simulate(r64, d64, tau)
        for _ in range(cfi):
            out = orc.simulate(r64, d64, tau)
        obs, rew, reset, _ = env.step(torch.tensor(a, device=env.device))
        torch.cuda.synchronize()
        keep = reset.cpu().numpy() == 0                      # reset envs were re-initialised by the second kernel
        rg = env.root_states.cpu().numpy()[keep]; dg = env.dof_state.cpu().numpy().reshape(n, nd, 2)[keep]
        assert np.isfinite(rg).all() and np.isfinite(dg).all() and torch.isfinite(obs["obs"]).all()
        n_cmp += int(keep.sum())
        assert np.abs(rg[:, :7] - r64[keep][:, :7]).max() < 3e-4, np.abs(rg[:, :7] - r64[keep][:, :7]).max()
        assert (np.abs(rg[:, 7:] - r64[keep][:, 7:]) / np.maximum(1, np.abs(r64[keep][:, 7:]))).max() < 1e-2
        assert np.abs(dg[..., 0] - d64[keep][..., 0]).max() < 3e-4
        tg = env.torques.cpu().numpy()[keep]
        assert np.abs(tg - tau[keep]).max() < 5e-2           # the last PD torque (Kp = 50, fp32 state)
        cg = env.contact_forces.cpu().numpy()[keep]
        co = out["contact_force"][keep]
        assert np.abs(cg - co).max() < 1e-2 * max(1.0, np.abs(co).max())
    assert n_cmp > 0.5 * n * steps


@pytest.mark.parametrize("terrain,n", [("plane", 256), ("trimesh", 256), ("trimesh", 4096), ("plane", 250)])
def test_fused_anymal_physics_equals_oracle_pd_loop(terrain, n):
    """anymal_physics_kernel (PD loop + 4+1 simulates, flat plane and curriculum height field) vs the oracle; N=4096 is the
    BASELINE.json size, N=250 is not a multiple of the 32 envs per block."""
    env = _make_anymal(n, terrain={"terrainType": terrain}, addNoise=False, pushRobots=False)
    rng = np.random.default_rng(3)
    env.step(torch.zeros(n, 12, device=env.device))           # the first step resets every env (reset_buf starts as ones)
    torch.cuda.synchronize()
    _anymal_check(env, 3, rng)


def test_cartpole_and_hand_baseline_sizes():
    """Cartpole 16384 and ShadowHand 4096 (BASELINE sizes) plus odd sizes: finite, resets happen, launch counts as documented."""
    for task, n, na in (("Cartpole", 16384, 1), ("Cartpole", 1001, 1), ("ShadowHand", 4096, 20), ("ShadowHand", 1001, 20)):
        env = _make(task, n)
        g = torch.Generator(device=env.device).manual_seed(0)
        c0 = env.sim.launch_count()
        for _ in range(8):
            obs, rew, reset, _ = env.step(2 * torch.rand((n, na), device=env.device, generator=g) - 1)
        torch.cuda.synchronize()
        assert env.sim.launch_count() == c0 + 8
        assert torch.isfinite(obs["obs"]).all() and torch.isfinite(rew).all()
        assert torch.isfinite(env.sim.root_state).all() and torch.isfinite(env.sim.dof_state).all()
        assert (env.progress_buf >= 0).all() and (env.progress_buf <= 8).all()


def test_hand_baseline_size_simulate_matches_oracle():
    """ShadowHand + cube at the BASELINE per-GPU size (4096 envs): one simulate from contact-rich states vs the oracle."""
    from tests.hand_common import settled_states
    from tests.test_gpu_parity import _hand_sim, _hand_load
    n = 4096
    m, obj, tendons, orc, root, dof, o, tgt = settled_states(n, 25, 5, threads=16)
    sim = _hand_sim(n, m, obj, tendons)
    _hand_load(sim, root, dof, o, tgt)
    rs = sim.root_state.cpu().numpy().astype(np.float64).reshape(n, 3, 13)
    r64 = np.ascontiguousarray(rs[:, 0]); o64 = np.ascontiguousarray(rs[:, 1])
    d64 = sim.dof_state.cpu().numpy().astype(np.float64).reshape(n, m.ndof, 2)
    t64 = sim.dof_target.cpu().numpy().astype(np.float64)
    sim.simulate(); torch.cuda.synchronize()
    orc.simulate(r64, d64, target=t64, obj=o64)
    rg = sim.root_state.cpu().numpy().astype(np.float64).reshape(n, 3, 13)
    dg = sim.dof_state.cpu().numpy().astype(np.float64).reshape(n, m.ndof, 2)
    assert np.abs(rg[:, 1, :3] - o64[:, :3]).max() < 5e-5
    assert np.abs(dg[..., 0] - d64[..., 0]).max() < 1e-4
    qerr = np.abs(dg[..., 1] - d64[..., 1]) / np.maximum(1.0, np.abs(d64[..., 1]))
    assert qerr.max() < 5e-3, qerr.max()
    sim.close()


# ------------------------------------------------------------------------------------ fast trigonometry
def test_fast_trig_build_is_bounded_against_exact_trig_build(tmp_path):
    """The product build evaluates joint rotations with __sincosf (B2G_FAST_TRIG=1).  Same library built with sincosf:
    one control step from states that include joint angles AT and beyond the limits (|q| up to 2.8 rad for the
    Humanoid knee) differs by < 2e-5 in base pose, < 1e-4 in joint positions (90 % below 1e-5, median below 1e-6) and < 5e-3 relative in joint velocities; after 30-step
    rollouts the median env is still within 1e-3 of its twin."""
    exact = os.path.join(ROOT, "isaacgymenvs_b200", "libb200gym_exacttrig.so")
    from isaacgymenvs_b200 import build as B
    if not os.path.exists(exact) or any(os.path.getmtime(d) > os.path.getmtime(exact) for d in B.DEPS):   # same ABI as the product build
        cmd = [os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc"), "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
               "--expt-relaxed-constexpr", "-Xcompiler", "-fPIC", "-shared", "-DB2G_FAST_TRIG=0", "-o", exact, B.SRC]
        subprocess.check_call(cmd)
    code = r'''
import os, sys, copy, numpy as np, torch
sys.path.insert(0, %r)
from isaacgymenvs_b200 import engine
from isaacgymenvs_b200.assets import load_compiled
G = (0.0, 0.0, -9.81)
out = {}
for name, zlo, zhi, ts in (("ant", 0.3, 0.8, 15.0), ("humanoid", 0.9, 1.6, 60.0)):
    m = copy.deepcopy(load_compiled(name))
    m.sensor_body = np.zeros(0, np.int32); m.sensor_pos = np.zeros((0, 3)); m.sensor_quat = np.zeros((0, 4))
    n = 512
    rng = np.random.default_rng(1)
    root = np.zeros((n, 13)); root[:, 2] = rng.uniform(zlo, zhi, size=n)
    q = rng.normal(size=(n, 4)) * np.array([0.3, 0.3, 0.3, 0.0]) + np.array([0, 0, 0, 1.0]); root[:, 3:7] = q / np.linalg.norm(q, axis=1, keepdims=True)
    root[:, 7:13] = rng.normal(size=(n, 6)) * 0.5
    lo, hi = m.lower[1:], m.upper[1:]
    u = rng.uniform(-0.05, 1.05, size=(n, m.ndof)); u[: n // 4] = np.round(u[: n // 4])        # a quarter of the envs sit exactly on a limit
    dof = np.stack([lo + (hi - lo) * u, rng.normal(size=(n, m.ndof))], -1)
    tau = rng.uniform(-1, 1, size=(n, m.ndof)) * ts
    sim = engine.Sim(m, n, 0.0166, 2, G)
    sim.root_state.copy_(torch.tensor(root, dtype=torch.float32)); sim.dof_state.copy_(torch.tensor(dof.reshape(-1, 2), dtype=torch.float32))
    sim.dof_actuation.copy_(torch.tensor(tau, dtype=torch.float32))
    sim.simulate(); torch.cuda.synchronize()
    out[name + "_root1"] = sim.root_state.cpu().numpy(); out[name + "_dof1"] = sim.dof_state.cpu().numpy()
    for k in range(29):
        sim.dof_actuation.copy_(torch.tensor(tau * np.sin(0.3 * k), dtype=torch.float32))
        sim.simulate()
    torch.cuda.synchronize()
    out[name + "_root30"] = sim.root_state.cpu().numpy(); out[name + "_dof30"] = sim.dof_state.cpu().numpy()
np.savez(sys.argv[1], **out)
''' % ROOT
    res = []
    for lib in ("", exact):
        out = str(tmp_path / f"trig_{int(bool(lib))}.npz")
        env_ = dict(os.environ)
        if lib:
            env_["B2G_LIB"] = lib
        subprocess.check_call([sys.executable, "-c", code, out], env=env_, cwd=ROOT)
        res.append(dict(np.load(out)))
    fast, ex = res
    for name in ("ant", "humanoid"):
        assert np.abs(fast[name + "_root1"][:, :7] - ex[name + "_root1"][:, :7]).max() < 2e-5
        d1f = fast[name + "_dof1"].reshape(512, -1, 2); d1e = ex[name + "_dof1"].reshape(512, -1, 2)
        dq1 = np.abs(d1f[..., 0] - d1e[..., 0])
        dv1 = np.abs(d1f[..., 1] - d1e[..., 1]) / np.maximum(1, np.abs(d1e[..., 1]))
        # measured on B200 (Ant): worst DOF 3.7e-5 rad / 2.0e-3 relative in velocity -- a foot pressed into the ground, where the
        # contact spring amplifies the 5e-7 absolute error of __sincosf; the 4 worst of 4096 DOFs reach 2.7e-5 rad; the bulk is
        # at rounding level
        assert dq1.max() < 1e-4 and np.quantile(dq1, 0.9) < 1e-5 and np.median(dq1) < 1e-6, (dq1.max(), np.quantile(dq1, 0.9), np.median(dq1))
        assert dv1.max() < 5e-3 and np.quantile(dv1, 0.9) < 5e-4 and np.median(dv1) < 5e-5, (dv1.max(), np.quantile(dv1, 0.9), np.median(dv1))
        # rollouts: contact-rich chaos amplifies any perturbation; the bulk of the envs must stay together
        dp = np.abs(fast[name + "_root30"][:, :3] - ex[name + "_root30"][:, :3]).max(1)
        assert np.isfinite(fast[name + "_root30"]).all()
        print(name, 'fast-vs-exact trig, 30 steps: median', np.median(dp), '90 %', np.quantile(dp, 0.9))
        assert np.median(dp) < 1e-3, np.median(dp)


# ------------------------------------------------------------------------------------ physical domain randomisation
@pytest.mark.parametrize("name,zlo,zhi,tscale,dt,sub", [("ant", 0.15, 0.8, 15.0, 0.0166, 2), ("anymal", 0.3, 0.9, 40.0, 0.005, 1),
                                                        ("humanoid", 0.9, 1.6, 60.0, 0.0166, 2)])
def test_per_env_physical_parameters_match_oracle(name, zlo, zhi, tscale, dt, sub):
    """B2G_T_ENV_MASS_SCALE / ENV_DOF_PROPS / ENV_FRICTION (vec_task.py:720-828 as parameter arrays): groups of envs with
    different link masses (the inertia follows: recomputeInertia, utils/dr_utils.py:62), joint damping / stiffness / limits and
    friction; each group equals the oracle run on a model with those values baked in (group 0 has every mass doubled).  Ant and
    ANYmal run on the four-chain kernels, the Humanoid on the generic sub-step."""
    from isaacgymenvs_b200 import engine
    from oracle.oracle import OracleSim
    base = copy.deepcopy(load_compiled(name))
    base.sensor_body = np.zeros(0, np.int32); base.sensor_pos = np.zeros((0, 3)); base.sensor_quat = np.zeros((0, 4))
    n, ng = 512, 4
    rng = np.random.default_rng(21)
    nl, nd = base.nl, base.ndof
    root = np.zeros((n, 13)); root[:, 0:2] = rng.normal(size=(n, 2)); root[:, 2] = rng.uniform(zlo, zhi, size=n)
    q = rng.normal(size=(n, 4)) * np.array([0.3, 0.3, 0.3, 0.0]) + np.array([0, 0, 0, 1.0]); root[:, 3:7] = q / np.linalg.norm(q, axis=1, keepdims=True)
    root[:, 7:13] = rng.normal(size=(n, 6)) * 0.5
    lo0 = np.where(base.limited[1:] > 0, base.lower[1:], -1.0); hi0 = np.where(base.limited[1:] > 0, base.upper[1:], 1.0)
    dof = np.stack([lo0 + (hi0 - lo0) * rng.uniform(-0.05, 1.05, size=(n, nd)), rng.normal(size=(n, nd))], -1)
    tau = rng.uniform(-1, 1, size=(n, nd)) * tscale
    sim = engine.Sim(base, n, dt, sub, G, ground_mu=1.0)
    assert sim.quad_ns() == {"ant": 2, "anymal": 3, "humanoid": 0}[name]
    sim.acquire(engine.T_NET_CONTACT)
    dev = sim.device
    ms_t = sim._bind(engine.T_ENV_MASS_SCALE, torch.ones(n, nl, device=dev))
    dp_t = sim._bind(engine.T_ENV_DOF_PROPS, torch.zeros(n, nd, 4, device=dev))
    fr_t = sim._bind(engine.T_ENV_FRICTION, torch.zeros(n, device=dev))
    sim.root_state.copy_(torch.tensor(root, dtype=torch.float32)); sim.dof_state.copy_(torch.tensor(dof.reshape(-1, 2), dtype=torch.float32))
    sim.dof_actuation.copy_(torch.tensor(tau, dtype=torch.float32))
    r64 = sim.root_state.cpu().numpy().astype(np.float64); d64 = sim.dof_state.cpu().numpy().astype(np.float64).reshape(n, nd, 2)
    t64 = sim.dof_actuation.cpu().numpy().astype(np.float64)
    lim = base.limited[1:] > 0
    cf = []
    for g in range(ng):
        ms = rng.uniform(0.5, 2.0, size=nl).astype(np.float32) if g else np.full(nl, 2.0, np.float32)
        dmp = (base.damping[1:] * rng.uniform(0.5, 1.5, size=nd) + 0.05 * g).astype(np.float32)
        stf = (base.stiffness[1:] * rng.uniform(0.5, 1.5, size=nd) + 0.5 * g).astype(np.float32)
        lo = np.where(lim, base.lower[1:] + rng.normal(0, 0.02, size=nd), -3e38).astype(np.float32)
        hi = np.where(lim, base.upper[1:] + rng.normal(0, 0.02, size=nd), 3e38).astype(np.float32)
        mu = np.float32(0.4 + 0.3 * g)
        sl = slice(g * n // ng, (g + 1) * n // ng)
        ms_t[sl] = torch.tensor(ms, device=dev); fr_t[sl] = float(mu)
        dp_t[sl] = torch.tensor(np.stack([dmp, stf, lo, hi], -1), device=dev)
        m = copy.deepcopy(base)
        m.mass = m.mass * ms.astype(np.float64)
        m.inertia = np.asarray(m.inertia, float) * ms.astype(np.float64)[:, None]      # recomputeInertia=True (vec_task.py:773): the inertia follows the mass
        m.damping = np.concatenate([[0.0], dmp.astype(np.float64)]); m.stiffness = np.concatenate([[0.0], stf.astype(np.float64)])
        m.lower = np.concatenate([[0.0], np.where(lim, lo.astype(np.float64), base.lower[1:])])
        m.upper = np.concatenate([[0.0], np.where(lim, hi.astype(np.float64), base.upper[1:])])
        m.cp_mu = np.full_like(np.asarray(m.cp_mu, float), float(mu))
        orc = OracleSim(m, dt, sub, G, ground_mu=1.0, threads=8)
        r = np.ascontiguousarray(r64[sl]); d = np.ascontiguousarray(d64[sl])
        cf.append(orc.simulate(r, d, np.ascontiguousarray(t64[sl]))["contact_force"])
        r64[sl] = r; d64[sl] = d
    sim.simulate(); torch.cuda.synchronize()
    rg = sim.root_state.cpu().numpy().astype(np.float64); dg = sim.dof_state.cpu().numpy().astype(np.float64).reshape(n, nd, 2)
    assert np.abs(rg[:, :7] - r64[:, :7]).max() < 2e-5
    dq = np.abs(dg[..., 0] - d64[..., 0])
    assert dq.max() < (5e-4 if name == "humanoid" else 2e-4) and np.quantile(dq, 0.999) < 3e-5, (dq.max(), np.quantile(dq, 0.999))
    qerr = np.abs(dg[..., 1] - d64[..., 1]) / np.maximum(1.0, np.abs(d64[..., 1]))
    assert qerr.max() < 4e-3 and np.quantile(qerr, 0.999) < 1e-3, (qerr.max(), np.quantile(qerr, 0.999))
    cg = sim.tensors[engine.T_NET_CONTACT].cpu().numpy().reshape(n, base.nb, 3)
    cb = np.concatenate(cf, 0)
    co = np.zeros_like(cb); first = {}
    for b in range(base.nb):                                   # the engine reports a link's contact force on the first body riding on it
        first.setdefault(int(base.body_link[b]), b)
        co[:, first[int(base.body_link[b])]] += cb[:, b]
    assert np.abs(cg - co).max() < 2e-3 * max(1.0, np.abs(co).max())
    sim.close()


def test_reset_done_resets_at_the_call():
    """VecTask.reset_done (vec_task.py:440-455): reset_idx of the flagged envs happens at the call -- state, counters and the
    flags change immediately, the reset Philox stream is the one the fused step uses, the next step does not reset again."""
    from oracle import tasks_np as T
    for task, nd in (("Ant", 8), ("Humanoid", 21), ("Cartpole", 2)):
        n = 64
        env = _make(task, n)
        assert (env.reset_buf == 1).all()
        obs, ids = env.reset_done()
        torch.cuda.synchronize()
        assert len(ids) == n and (env.reset_buf == 0).all() and (env.progress_buf == 0).all() and (env.reset_count == 1).all()
        q = env.dof_state.view(n, nd, 2)[..., 0].cpu().numpy(); qd = env.dof_state.view(n, nd, 2)[..., 1].cpu().numpy()
        if task != "Cartpole":
            lo, hi = env.dof_limits_lower_np, env.dof_limits_upper_np
            init = np.where(lo > 0, lo, np.where(hi < 0, hi, 0)).astype(f32)
            for e in (0, n - 1):
                u = T.reset_uniforms(42, e, 0, 2 * nd)
                assert np.allclose(q[e], np.clip(init + (f32(0.4) * u[:nd] + f32(-0.2)), lo, hi), atol=1e-7)
                assert np.allclose(qd[e], f32(0.2) * u[nd:] + f32(-0.1), atol=1e-7)
            assert np.allclose(env.root_states.cpu().numpy(), env.initial_root_states.cpu().numpy())
            assert torch.equal(env.potentials, env.prev_potentials)
        c0 = env.sim.launch_count()
        env.step(torch.zeros(n, env.num_acts, device=env.device))
        torch.cuda.synchronize()
        assert env.sim.launch_count() == c0 + 1 and (env.reset_count == 1).all() and (env.progress_buf == 1).all()
        _, ids2 = env.reset_done()                                       # nothing flagged: no launch
        assert len(ids2) == int(env.reset_buf.sum().item()) and env.sim.launch_count() == c0 + 1 + (1 if len(ids2) else 0)
    for task, na in (("AnymalTerrain", 12), ("ShadowHand", 20)):
        n = 64
        env = _make(task, n)
        env.reset_done()
        torch.cuda.synchronize()
        assert (env.progress_buf == 0).all() and (env.reset_count == 1).all()
        assert torch.isfinite(env.sim.root_state).all() and torch.isfinite(env.sim.dof_state).all()
        for _ in range(3):
            obs, rew, reset, _ = env.step(torch.zeros(n, na, device=env.device))
        torch.cuda.synchronize()
        assert torch.isfinite(obs["obs"]).all() and (env.reset_count >= 1).all()


@pytest.mark.parametrize("n,K,ep_len", [(256, 12, 5), (16384, 6, 1000), (1000, 4, 3)])
def test_rollout_equals_k_single_steps(n, K, ep_len):
    """b2g_task_rollout (one launch, state on chip across the K steps) == K x VecTask.step() on every output of every step and
    on every bound tensor afterwards; short episodes put time-out resets (and their Philox draws) inside the rollout.
    n = 1000 is not whole tiles of 16: the documented K-single-steps fallback, same contract."""
    a_env = _make("Ant", n, episodeLength=ep_len)
    b_env = _make("Ant", n, episodeLength=ep_len)
    g = torch.Generator(device="cuda:0"); g.manual_seed(7)
    acts = (torch.rand((K, n, a_env.num_acts), device="cuda:0", generator=g) * 2 - 1) * 1.2          # beyond the clamp too
    ref_o, ref_r, ref_d, ref_t = [], [], [], []
    for k in range(K):
        od, r, d, info = a_env.step(acts[k])
        ref_o.append(od["obs"].clone()); ref_r.append(r.clone()); ref_d.append(d.clone()); ref_t.append(info["time_outs"].clone())
    c0 = b_env.sim.launch_count()
    obs, rew, done, tout = b_env.rollout(acts)
    torch.cuda.synchronize()
    if n % 16 == 0:
        assert b_env.sim.launch_count() == c0 + 1
    # The two paths are different kernels: their arithmetic agrees to rounding, not bit for bit, and the joint-limit law is
    # discontinuous where a joint crosses its limit at speed (the damper engages abruptly, DESIGN.md section 7) -- an env that
    # does so inside the rollout amplifies a 1-ulp difference to O(1) within a step (measured: 7 of 16384 envs in 6 steps).
    # So: every env identical to 2e-4 up to a 0.2 % share of such outliers, flags identical on all the others.
    dobs = (obs - torch.stack(ref_o)).abs().amax(dim=(0, 2))                     # worst entry per env
    off = dobs >= 2e-4
    if off.any():
        print("rollout != steps (beyond 2e-4) in", int(off.sum()), "of", n, "envs:", off.nonzero().flatten()[:16].tolist())
    assert off.float().mean().item() <= 0.002, int(off.sum())
    ok = ~off
    assert torch.equal(done[:, ok], torch.stack(ref_d)[:, ok]) and torch.equal(tout[:, ok], torch.stack(ref_t).bool()[:, ok])
    assert done.sum().item() > 0 or ep_len > K
    # (derived quantities amplify what the observation scales down: the progress reward is a position difference / dt = x60,
    # joint velocities enter the observation x0.2 -- hence the looser bounds on them for envs whose observations agree to 2e-4)
    assert (rew - torch.stack(ref_r)).abs()[:, ok].max().item() < 2e-2
    for name, tol in (("root_states", 2e-3), ("dof_state", 2e-3), ("potentials", 2e-2), ("prev_potentials", 2e-2), ("obs_buf", 2e-4),
                      ("rew_buf", 2e-2), ("vec_sensor_tensor", 2e-2)):
        x, y = getattr(a_env, name), getattr(b_env, name)
        d = (x - y).abs().reshape(n, -1).amax(1)
        assert d[ok].max().item() < tol, (name, d[ok].max().item())
    for name in ("progress_buf", "reset_buf", "reset_count"):
        assert torch.equal(getattr(a_env, name)[ok], getattr(b_env, name)[ok]), name
    # and the env keeps stepping normally afterwards
    z = torch.zeros(n, a_env.num_acts, device="cuda:0")
    oa, ob = a_env.step(z)[0]["obs"], b_env.step(z)[0]["obs"]
    assert ((oa - ob).abs().amax(1) >= 3e-4).float().mean().item() <= 0.003


# ------------------------------------------------------------------------------------ self-collision (collision filter 0)
def _sphere_overlap(m, orc, root, dof):
    """deepest overlap (m) between contact spheres of links that may collide (model.self_pairs), per env"""
    from oracle import tasks_np as T
    cpb = np.array(m.cp_body)
    bs = orc.body_states(root, dof)
    off_p = np.asarray(m.body_pos, f32)[cpb]; off_q = np.asarray(m.body_quat, f32)[cpb]
    loc = T.quat_rotate_inverse(off_q, np.asarray(m.cp_pos, f32) - off_p)
    n, ncp = bs.shape[0], len(cpb)
    wp = bs[:, cpb, 0:3].astype(f32) + T.quat_rotate(bs[:, cpb, 3:7].astype(f32).reshape(-1, 4), np.tile(loc, (n, 1))).reshape(n, ncp, 3)
    rr = (np.asarray(m.cp_radius)[:, None] + np.asarray(m.cp_radius)[None, :]).astype(f32)
    d = np.linalg.norm(wp[:, :, None, :] - wp[:, None, :, :], axis=-1)
    return np.where(np.asarray(m.self_pairs)[None] > 0, rr[None] - d, -1.0).max(axis=(1, 2))


def test_self_collision_engine_matches_oracle():
    """Link-link contact (humanoid.py:194 collision filter 0) in the generic sub-step against the oracle's restatement: one
    control step from 1024 random Humanoid configurations -- joints anywhere inside their limits, so most states start with
    limbs touching or overlapping (arms in the torso, legs crossed), some also on the ground."""
    from oracle.oracle import OracleSim
    from isaacgymenvs_b200 import engine
    from isaacgymenvs_b200.importer.model import enable_self_collision
    m = copy.deepcopy(load_compiled("humanoid"))
    m.angular_damping, m.max_angular_velocity = 0.01, 100.0
    enable_self_collision(m)
    n = 1024
    rng = np.random.default_rng(5)
    root = np.zeros((n, 13)); root[:, 2] = rng.uniform(0.9, 2.5, size=n)
    q = rng.normal(size=(n, 4)) * np.array([0.4, 0.4, 0.4, 0.0]) + np.array([0, 0, 0, 1.0]); root[:, 3:7] = q / np.linalg.norm(q, axis=1, keepdims=True)
    root[:, 7:13] = rng.normal(size=(n, 6)) * 0.5
    lo, hi = m.lower[1:], m.upper[1:]
    dof = np.stack([rng.uniform(lo, hi, size=(n, m.ndof)), rng.normal(size=(n, m.ndof)) * 2.0], -1)
    tau = rng.uniform(-1, 1, size=(n, m.ndof)) * np.asarray(m.actuator_gear)[None] * 0.3
    orc = OracleSim(m, 0.0166, 2, G, threads=8)
    dep = _sphere_overlap(m, orc, root, dof)
    assert (dep > 0.0).mean() > 0.15, (dep > 0).mean()              # the sample really exercises link-link contact
    sim = engine.Sim(m, n, 0.0166, 2, G)
    assert sim.quad_ns() == 0
    nc = sim.acquire(engine.T_NET_CONTACT)
    sim.root_state.copy_(torch.tensor(root, dtype=torch.float32)); sim.dof_state.copy_(torch.tensor(dof.reshape(-1, 2), dtype=torch.float32))
    sim.dof_actuation.copy_(torch.tensor(tau, dtype=torch.float32))
    r64 = sim.root_state.cpu().numpy().astype(np.float64); d64 = sim.dof_state.cpu().numpy().astype(np.float64).reshape(n, m.ndof, 2)
    t64 = sim.dof_actuation.cpu().numpy().astype(np.float64)
    sim.simulate(); torch.cuda.synchronize()
    out = orc.simulate(r64, d64, t64)
    rg = sim.root_state.cpu().numpy().astype(np.float64); dg = sim.dof_state.cpu().numpy().astype(np.float64).reshape(n, m.ndof, 2)
    assert np.isfinite(rg).all() and np.isfinite(dg).all()
    # stiff contacts between light limbs amplify fp32 round-off more than the ground contact does: layered bounds
    dp = np.abs(rg[:, :7] - r64[:, :7]).max(1)
    assert np.quantile(dp, 0.99) < 5e-5 and dp.max() < 1e-3, (np.quantile(dp, 0.99), dp.max())
    dq = np.abs(dg[..., 0] - d64[..., 0])
    assert np.quantile(dq, 0.99) < 1e-4 and dq.max() < 5e-3, (np.quantile(dq, 0.99), dq.max())
    qerr = np.abs(dg[..., 1] - d64[..., 1]) / np.maximum(1.0, np.abs(d64[..., 1]))
    assert np.quantile(qerr, 0.99) < 2e-3 and np.median(qerr) < 1e-4, (np.quantile(qerr, 0.99), np.median(qerr))
    # the engine reports the contact force of a LINK on the first body riding on it (head -> torso, hand -> lower arm are welded
    # bodies of one link: DevModel::link_body); the oracle reports per body -- sum the oracle's over each link before comparing
    cg = nc.cpu().numpy().reshape(n, m.nb, 3); co = np.zeros_like(out["contact_force"])
    first = {}
    for b in range(m.nb):
        first.setdefault(int(m.body_link[b]), b)
        co[:, first[int(m.body_link[b])]] += out["contact_force"][:, b]
    cerr = np.abs(cg - co).max(axis=(1, 2)) / np.maximum(1.0, np.abs(co).max(axis=(1, 2)))
    assert np.quantile(cerr, 0.99) < 1e-2 and np.median(cerr) < 1e-3, (np.quantile(cerr, 0.99), np.median(cerr))
    # and the same model without the flag is a different trajectory (the contact is really applied)
    m2 = copy.deepcopy(m); m2.self_collide = False
    s2 = engine.Sim(m2, n, 0.0166, 2, G)
    s2.root_state.copy_(torch.tensor(root, dtype=torch.float32)); s2.dof_state.copy_(torch.tensor(dof.reshape(-1, 2), dtype=torch.float32))
    s2.dof_actuation.copy_(torch.tensor(tau, dtype=torch.float32))
    s2.simulate(); torch.cuda.synchronize()
    assert (np.abs(s2.dof_state.cpu().numpy().reshape(n, m.ndof, 2)[..., 1] - dg[..., 1]).max(1) > 0.1).mean() > 0.1
    sim.close(); s2.close()


def test_humanoid_limbs_do_not_interpenetrate():
    """env.selfCollision=True: the Humanoid task collides its links with each other like the reference (collision filter 0).
    Random-action rollout: the share of sampled env-states with two non-neighbour bodies overlapping by more than 1 cm is
    at most half of what it is without it (a soft penalty contact: gains bounded by the stability of the half-explicit
    coupling), which is > 15 % -- the default, which must announce itself with an UnmodelledPhysicsWarning, as the
    four-chain ANYmal kernels (no link-link contact) do."""
    import warnings
    from oracle.oracle import OracleSim
    from isaacgymenvs_b200 import engine
    share = {}
    for on in (True, False):
        engine._warned.discard("Humanoid")
        with warnings.catch_warnings(record=True) as rec:
            warnings.simplefilter("always")
            env = _make("Humanoid", 1024, selfCollision=on)
        warned = any(issubclass(w.category, engine.UnmodelledPhysicsWarning) for w in rec)
        assert warned == (not on)
        m = copy.deepcopy(env.model)
        if not on:
            from isaacgymenvs_b200.importer.model import enable_self_collision
            enable_self_collision(m); m.self_collide = False            # pair table for the measurement only
        assert bool(getattr(env.model, "self_collide", False)) == on
        orc = OracleSim(m, 0.0166, 2, G)
        g = torch.Generator(device="cuda:0"); g.manual_seed(3)
        hits = samples = 0; worst = 0.0
        for k in range(120):
            env.step(torch.rand((1024, env.num_acts), device="cuda:0", generator=g) * 2 - 1)
            if k % 10 != 9:
                continue
            torch.cuda.synchronize()
            dep = _sphere_overlap(m, orc, env.root_states.cpu().numpy().astype(np.float64), env.dof_state.cpu().numpy().astype(np.float64).reshape(1024, -1, 2))
            hits += int((dep > 0.01).sum()); samples += 1024; worst = max(worst, float(dep.max()))
        assert torch.isfinite(env.root_states).all() and torch.isfinite(env.dof_state).all()
        share[on] = hits / samples
        print(f"Humanoid, random actions, self-collision {'on' if on else 'off'}: {hits}/{samples} sampled env-states overlap > 1 cm "
              f"({100.0 * hits / samples:.1f} %), deepest {worst * 100:.1f} cm")
    assert share[True] < 0.5 * share[False] and share[False] > 0.15, share
    engine._warned.discard("AnymalTerrain")
    with warnings.catch_warnings(record=True) as rec:
        warnings.simplefilter("always")
        _make_anymal(64)
    assert any(issubclass(w.category, engine.UnmodelledPhysicsWarning) for w in rec)


# ---------------------------------------------------------------------------------------------
# random forces on the object (env.forceScale > 0, shadow_hand.py:69-72,196-201,616,642,700-709)
def test_hand_random_object_forces_match_reference_golden():
    """The fused ShadowHand step with forceScale = 2 (no physics: controlFrequencyInv = 0) from the inputs of golden case "f":
    decay of the carried force, zeroing + new probability on reset, redraw where rand < random_force_prob -- against the
    reference's own pre_physics_step (tests/golden/make_golden_hand.py --force)."""
    from tests.hand_common import force_constants
    from tests.test_gpu_parity import _hand_env, GOLD
    gold = np.load(os.path.join(GOLD, "shadow_hand_force.npz"))
    gi = lambda k: gold[f"f_in_{k}"]
    go = lambda k: gold[f"f_out_{k}"]
    n = gi("reset").shape[0]
    env = _hand_env(n, "f", "full_state", forceScale=float(gold["force_scale"]), forceProbRange=[float(v) for v in gold["force_prob_range"]])
    fc = force_constants(gold)
    assert env.sim.task.force_scale == fc["force_scale"] and env.sim.task.force_decay_factor == np.float32(fc["force_decay_factor"])
    assert abs(float(env.object_rb_masses[0]) - fc["obj_mass"]) < 1e-9
    dev = env.device
    t = lambda a, dt=torch.float32: torch.tensor(np.asarray(a), dtype=dt, device=dev)
    env.root_state_tensor.copy_(t(gi("root")))
    env.initial_root_states.view(n, 3, 13)[:, 1].copy_(t(gi("object_init")))
    env.initial_root_states.view(n, 3, 13)[:, 2].copy_(t(gi("goal_init")))
    env.dof_state.copy_(t(gi("dof_state")))
    env.prev_targets.copy_(t(gi("prev_targets"))); env.cur_targets.copy_(t(gi("cur_targets")))
    env.goal_states.copy_(t(gi("goal_states")))
    env.vec_sensor_tensor.copy_(t(gi("sensors"))); env.dof_force_tensor.copy_(t(gi("dof_force")))
    env.reset_buf.copy_(t(gi("reset"), torch.long)); env.reset_goal_buf.copy_(t(gi("reset_goal"), torch.long))
    env.progress_buf.copy_(t(gi("progress"), torch.long)); env.successes.copy_(t(gi("successes")))
    env._cons[0] = float(gi("cons")[0])
    env.reset_count.copy_(t(gi("reset_count"), torch.int32)); env.goal_reset_count.copy_(t(gi("goal_reset_count"), torch.int32))
    env.object_rb_forces.copy_(t(gi("obj_force"))); env.random_force_prob.copy_(t(gi("force_prob")))
    env.step(t(gi("actions")))
    torch.cuda.synchronize()
    c = lambda x: x.detach().cpu().numpy()
    # the same envs drew a new force; values to fp32 round-off of log / sqrt / cos (Box-Muller) and exp
    drew_ref = (go("obj_force") != gi("obj_force") * np.float32(fc["force_decay_factor"])).any(1)
    drew_gpu = (c(env.object_rb_forces) != gi("obj_force") * np.float32(fc["force_decay_factor"])).any(1)
    assert np.array_equal(drew_ref | (gi("reset") != 0), drew_gpu | (gi("reset") != 0)) and drew_ref.sum() > 100
    np.testing.assert_allclose(c(env.object_rb_forces), go("obj_force"), rtol=2e-5, atol=2e-7)
    np.testing.assert_allclose(c(env.random_force_prob), go("force_prob"), rtol=2e-6)
    assert np.array_equal(c(env.rb_forces)[:, env.model.nb], c(env.object_rb_forces)) and float(env.rb_forces[:, :env.model.nb].abs().max()) == 0.0
    # everything else of the step is what it is without forces
    np.testing.assert_allclose(c(env.root_state_tensor), go("root"), rtol=0, atol=1e-6)
    np.testing.assert_allclose(c(env.rew_buf), go("rew"), rtol=3e-6, atol=3e-5)
    assert np.array_equal(c(env.reset_buf), go("reset")) and np.array_equal(c(env.progress_buf), go("progress"))
    # reset_done (b2g_reset_flagged) zeroes the force and redraws the probability from the reset stream too
    env.reset_buf.fill_(1); before = c(env.random_force_prob).copy()
    env.reset_done(); torch.cuda.synchronize()
    assert float(env.object_rb_forces.abs().max()) == 0.0 and (c(env.random_force_prob) != before).mean() > 0.9
    lo, hi = [float(v) for v in gold["force_prob_range"]]
    assert (c(env.random_force_prob) >= lo * (1 - 1e-5)).all() and (c(env.random_force_prob) <= hi * (1 + 1e-5)).all()
    env.sim.close()


def test_hand_object_force_physics_matches_oracle():
    """gym.apply_rigid_body_force_tensors(..., LOCAL_SPACE) on the object: one gym.simulate() with a force bound to OBJ_FORCE
    against the oracle given the same force; and a cube in free flight accelerates by g + R f / m."""
    from isaacgymenvs_b200 import engine
    from tests.hand_common import settled_states, DT
    from tests.test_gpu_parity import _hand_sim, _hand_load
    n = 256
    m, obj, tendons, orc, root, dof, o, tgt = settled_states(n, 40, 7)
    rng = np.random.default_rng(3)
    o[n // 2:, 2] += 1.0                                       # half of the cubes in free flight
    f = (rng.normal(size=(n, 3)) * obj["mass"] * 20.0).astype(np.float32)
    sim = _hand_sim(n, m, obj, tendons)
    _hand_load(sim, root, dof, o, tgt)
    of = sim._bind(engine.T_OBJ_FORCE, torch.tensor(f, device=sim.device))
    rs = sim.root_state.cpu().numpy().astype(np.float64).reshape(n, 3, 13)
    r64 = np.ascontiguousarray(rs[:, 0]); o64 = np.ascontiguousarray(rs[:, 1]); o_in = o64.copy()
    d64 = sim.dof_state.cpu().numpy().astype(np.float64).reshape(n, m.ndof, 2)
    t64 = sim.dof_target.cpu().numpy().astype(np.float64)
    r2, d2, o_no = r64.copy(), d64.copy(), o64.copy()
    sim.simulate(); torch.cuda.synchronize()
    orc.simulate(r64, d64, target=t64, obj=o64, obj_force=f.astype(np.float64))
    rg = sim.root_state.cpu().numpy().astype(np.float64).reshape(n, 3, 13)
    assert np.abs(rg[:, 1, :3] - o64[:, :3]).max() < 5e-5
    verr = np.abs(rg[:, 1, 7:] - o64[:, 7:]) / np.maximum(1.0, np.abs(o64[:, 7:]))
    assert verr.max() < 5e-3, verr.max()
    # the force matters (the oracle without it lands elsewhere) ...
    orc.simulate(r2, d2, target=t64, obj=o_no)
    assert np.abs(o_no[:, 7:10] - o64[:, 7:10]).max() > 0.05
    # ... and in free flight it is exactly Newton: dv = (g + R f / m) dt  (the body-frame force turns with the cube: tolerance for the spin)
    from isaacgymenvs_b200.importer import rot
    fl = slice(n // 2, n)
    R = np.stack([rot.quat_to_mat(q) for q in o_in[fl, 3:7]])
    dv = (rg[fl, 1, 7:10] - o_in[fl, 7:10]) / DT
    want = np.array([0.0, 0.0, -9.81]) + np.einsum("nij,nj->ni", R, f[fl].astype(np.float64)) / obj["mass"]
    assert np.abs(dv - want).max() < 0.05 * np.abs(want).max()
    sim.close()


# ---------------------------------------------------------------------------------------------
# ShadowHand objectType egg / pen (shadow_hand.py:84-99): the free object as a rounded box
@pytest.mark.parametrize("name", ["pen", "egg"])
def test_hand_rounded_object_simulate_matches_oracle(name):
    """One gym.simulate() from contact-rich states of the hand with the pen (capsule) / the egg (spheroid carried as a capsule):
    engine against oracle, same tolerances as the cube's test (tests/test_gpu_parity.py::test_hand_object_simulate_matches_oracle)."""
    from isaacgymenvs_b200 import engine
    from tests.hand_common import settled_states
    from tests.test_gpu_parity import _hand_sim, _hand_load
    n = 512
    m, obj, tendons, orc, root, dof, o, tgt = settled_states(n, 40, 9, obj_name=name)
    o[: n // 8, 2] = obj["round"] + 0.3 * obj["half"][2] + 0.001            # some on the ground, tilted
    sim = _hand_sim(n, m, obj, tendons)
    _hand_load(sim, root, dof, o, tgt)
    rs = sim.root_state.cpu().numpy().astype(np.float64).reshape(n, 3, 13)
    r64 = np.ascontiguousarray(rs[:, 0]); o64 = np.ascontiguousarray(rs[:, 1]); o_in = o64.copy()
    d64 = sim.dof_state.cpu().numpy().astype(np.float64).reshape(n, m.ndof, 2)
    t64 = sim.dof_target.cpu().numpy().astype(np.float64)
    sim.simulate(); torch.cuda.synchronize()
    out = orc.simulate(r64, d64, target=t64, obj=o64)
    rg = sim.root_state.cpu().numpy().astype(np.float64).reshape(n, 3, 13)
    dg = sim.dof_state.cpu().numpy().astype(np.float64).reshape(n, m.ndof, 2)
    assert np.isfinite(rg).all() and np.isfinite(o64).all()
    # objects knocked into a fast tumble sit on the angular-speed clamp, where the explicitly integrated gyroscopic term of the
    # slender pen amplifies round-off: compare the ones below half the clamp (the bulk), bound the rest
    calm = np.linalg.norm(o_in[:, 10:13], axis=1) < 30.0
    assert calm.mean() > 0.8
    assert np.abs(rg[calm, 1, :3] - o64[calm, :3]).max() < 5e-5 and np.abs(rg[:, 1, :3] - o64[:, :3]).max() < 2e-3
    qd = np.minimum(np.abs(rg[:, 1, 3:7] - o64[:, 3:7]).max(-1), np.abs(rg[:, 1, 3:7] + o64[:, 3:7]).max(-1))
    verr = np.abs(rg[:, 1, 7:] - o64[:, 7:]) / np.maximum(1.0, np.abs(o64[:, 7:]))
    if name == "pen":
        # spin about the pen's own axis: inertia 1.3e-6 kg m^2 against m |c|^2 ~ 1e-2 in the engine's 6x6 solve about the root
        # origin -- fp32 leaves ~1e-3 relative accuracy for that one component when contact friction spins the pen up.  The
        # centre-of-mass motion and the bulk of the orientations are as tight as the cube's; the axial tail is bounded.
        assert np.percentile(qd[calm], 90) < 2e-4 and qd[calm].max() < 2e-2, (np.percentile(qd[calm], 90), qd[calm].max())
        assert verr[calm][:, :3].max() < 5e-3 and np.percentile(verr[calm][:, 3:].max(-1), 90) < 5e-3, (verr[calm][:, :3].max(), np.percentile(verr[calm][:, 3:].max(-1), 90))
    else:
        assert qd[calm].max() < 2e-4, qd[calm].max()
        assert verr[calm].max() < 5e-3, verr[calm].max()
    assert np.linalg.norm(rg[:, 1, 10:13], axis=1).max() <= 64.0 * (1 + 1e-5)
    assert np.abs(dg[..., 0] - d64[..., 0]).max() < 1e-4
    qerr = np.abs(dg[..., 1] - d64[..., 1]) / np.maximum(1.0, np.abs(d64[..., 1]))
    assert qerr.max() < 5e-3, qerr.max()
    sg = sim.tensors[engine.T_FORCE_SENSOR].cpu().numpy().reshape(n, -1, 6)
    assert np.abs(out["sensor"]).max() > 0.05                                            # the fingertips do touch the object
    assert np.abs(sg - out["sensor"]).max() < 5e-3 * max(1.0, np.abs(out["sensor"]).max())
    # the object was in contact in a good share of the envs (not a free-flight test)
    g_only = o_in[:, 7:10] + np.array([0, 0, -9.81]) * 0.01667
    assert (np.abs(o64[:, 7:10] - g_only).max(-1) > 1e-3).mean() > 0.3
    sim.close()


@pytest.mark.parametrize("name", ["pen", "egg"])
def test_hand_env_with_egg_and_pen_runs(name):
    """env.objectType egg / pen through make(): the object shape reaches the engine, the step stays finite, objects that fall
    are reset, and the pen doubles the success tolerance (ignore_z_rot, shadow_hand.py:758-759)."""
    env = _make("ShadowHand", 256, objectType=name)
    assert env.object_type == name and env.ignore_z == (name == "pen")
    assert env.sim.task.success_tolerance == np.float32(0.1 * (2.0 if name == "pen" else 1.0))
    g = torch.Generator(device=env.device).manual_seed(1)
    nres = 0
    for k in range(120):
        obs, rew, reset, extras = env.step(2 * torch.rand(256, 20, device=env.device, generator=g) - 1)
        nres += int(reset.sum())
    torch.cuda.synchronize()
    assert torch.isfinite(obs["obs"]).all() and torch.isfinite(rew).all() and torch.isfinite(env.root_state_tensor).all()
    assert nres > 0                                              # random actions drop the object sooner or later
    z = env.root_state_tensor.view(256, 3, 13)[:, 1, 2]
    assert float(z.min()) > -0.01                                # nothing tunnels through the ground
    env.sim.close()
