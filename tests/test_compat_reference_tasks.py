"""The compatibility path on CPU: the reference's UNMODIFIED task files (loaded from
/root/reference, never copied) import against the `isaacgym` shim and run their own Python hooks --
create_sim / pre_physics_step / post_physics_step / reset_idx / jit obs+reward -- through the
hook-style VecTask.  The engine itself needs a GPU, so here `engine.Sim` is replaced by a stand-in
with the same tensors whose `simulate()` integrates nothing: what is tested is the API surface, the
tensor-view contracts (aliasing, indexed setters) and that the reference code runs unmodified."""
import os
import sys
import types
import numpy as np
import pytest
import torch

from tests.conftest import needs_reference, REFERENCE


class _FakeSim:
    def __init__(self, model, num_envs, dt, substeps, gravity=(0, 0, -9.81), ground_mu=1.0, device="cpu", ext=None, **kw):
        from isaacgymenvs_b200 import engine as E
        self.model, self.num_envs, self.ext, self.kw = model, num_envs, ext, kw
        self.actors_per_env = int(ext.actors_per_env) if ext is not None else 1
        self.nd, self.nb, self.ns = model.ndof, model.nb, len(model.sensor_body)
        self.root_state = torch.zeros(num_envs * self.actors_per_env, 13); self.root_state[:, 6] = 1
        self.dof_state = torch.zeros(num_envs * max(self.nd, 1), 2)
        self.dof_actuation = torch.zeros(num_envs, max(self.nd, 1)); self.dof_target = torch.zeros_like(self.dof_actuation)
        self.tensors, self.E, self.steps = {}, E, 0

    def acquire(self, slot):
        E, N = self.E, self.num_envs
        shape = {E.T_RIGID_BODY_STATE: (N * (self.nb + self.actors_per_env - 1), 13), E.T_FORCE_SENSOR: (N * max(self.ns, 1), 6),
                 E.T_DOF_FORCE: (N * max(self.nd, 1),), E.T_NET_CONTACT: (N * self.nb, 3)}[slot]
        return self.tensors.setdefault(slot, torch.zeros(*shape))

    def _bind(self, slot, t):
        self.tensors[slot] = t
        return t

    def simulate(self):
        self.steps += 1
        self.seen_obj_force = self.tensors[self.E.T_OBJ_FORCE].clone() if self.E.T_OBJ_FORCE in self.tensors else None

    def refresh_rigid_body_state(self):
        return self.acquire(self.E.T_RIGID_BODY_STATE)


@pytest.fixture
def compat_cpu(monkeypatch):
    from isaacgymenvs_b200 import compat, engine
    from isaacgymenvs_b200.compat import vec_task_hooks
    saved = {k: v for k, v in sys.modules.items() if k.startswith("isaacgym")}
    for k in list(saved):
        if k.startswith("isaacgymenvs.") or k in ("isaacgym", "isaacgymenvs") or k.startswith("isaacgym."):
            if not k.startswith("isaacgymenvs_b200"):
                del sys.modules[k]
    compat.install(reference_root=REFERENCE)
    monkeypatch.setattr(engine, "Sim", _FakeSim)
    vec_task_hooks.reset_sim_singleton()
    yield
    vec_task_hooks.reset_sim_singleton()
    for k in list(sys.modules):
        if (k == "isaacgym" or k.startswith("isaacgym.") or k == "isaacgymenvs" or k.startswith("isaacgymenvs.")):
            del sys.modules[k]
    sys.modules.update({k: v for k, v in saved.items() if not k.startswith("isaacgymenvs_b200")})


def _cfg(task, n):
    from isaacgymenvs_b200 import config
    c = config.load_reference_cfg(os.path.join(REFERENCE, "isaacgymenvs", "cfg"), task, {"pipeline": "cpu", "sim_device": "cpu", "rl_device": "cpu"})
    t = c["task"]
    t["env"]["numEnvs"] = n
    t["sim"]["use_gpu_pipeline"] = False
    return t


@needs_reference
@pytest.mark.parametrize("task,module,cls,nobs,nact", [("Ant", "ant", "Ant", 60, 8), ("Humanoid", "humanoid", "Humanoid", 108, 21),
                                                       ("Cartpole", "cartpole", "Cartpole", 4, 1)])
def test_unmodified_reference_task_runs_on_the_shim(compat_cpu, task, module, cls, nobs, nact):
    import importlib
    mod = importlib.import_module(f"isaacgymenvs.tasks.{module}")          # the reference's own file
    assert os.path.realpath(mod.__file__).startswith(REFERENCE)
    n = 16
    env = getattr(mod, cls)(cfg=_cfg(task, n), rl_device="cpu", sim_device="cpu", graphics_device_id=-1, headless=True,
                            virtual_screen_capture=False, force_render=False)
    assert env.num_obs == nobs and env.num_acts == nact and env.obs_buf.shape == (n, nobs)
    sim = env.sim.engine
    # state tensors are views of the simulator's memory (ant.py:93-95)
    assert env.dof_state.data_ptr() == sim.dof_state.data_ptr()
    torch.manual_seed(0)
    obs, rew, reset, extras = env.step(2 * torch.rand(n, nact) - 1)      # first step resets every env (reset_buf starts as ones)
    assert sim.steps == env.control_freq_inv
    assert obs["obs"].shape == (n, nobs) and torch.isfinite(obs["obs"]).all() and torch.isfinite(rew).all()
    assert (env.progress_buf == 0).all() and "time_outs" in extras
    if task != "Cartpole":
        # reset_idx wrote the randomised joint state through its views and the root through the indexed setter
        lo, hi = env.dof_limits_lower, env.dof_limits_upper
        assert ((env.dof_pos >= lo - 1e-6) & (env.dof_pos <= hi + 1e-6)).all() and env.dof_pos.abs().sum() > 0
        assert torch.allclose(sim.root_state, env.initial_root_states)
        assert abs(float(sim.root_state[0, 2]) - (0.44 if task == "Ant" else 1.34)) < 1e-6
        # forces reached the actuation tensor: action * gear (ant.py:283-285)
        assert sim.dof_actuation.abs().max() > 1.0
    obs2, rew2, reset2, _ = env.step(torch.zeros(n, nact))
    assert (env.progress_buf == 1).all()


@needs_reference
def test_unmodified_reference_shadow_hand_runs_on_the_shim(compat_cpu):
    """Three actors per env (hand, cube, goal marker), tendon properties, actor-indexed setters, the 211-d full_state
    observation: the reference's own shadow_hand.py drives the shim unmodified."""
    import importlib
    mod = importlib.import_module("isaacgymenvs.tasks.shadow_hand")
    assert os.path.realpath(mod.__file__).startswith(REFERENCE)
    n = 8
    env = mod.ShadowHand(cfg=_cfg("ShadowHand", n), rl_device="cpu", sim_device="cpu", graphics_device_id=-1, headless=True,
                         virtual_screen_capture=False, force_render=False)
    sim = env.sim.engine
    assert env.num_obs == 211 and env.num_acts == 20 and env.num_shadow_hand_dofs == 24 and env.num_shadow_hand_actuators == 20
    # the engine was created with the multi-actor extras the task's calls imply
    ext = sim.ext
    assert ext.actors_per_env == 3 and ext.obj_actor == 1 and ext.nten == 4 and abs(ext.ten_k - 30.0) < 1e-6 and abs(ext.ten_d - 0.1) < 1e-6
    assert abs(ext.obj_mass - 0.070875) < 1e-6 and [round(v, 4) for v in ext.obj_half] == [0.025, 0.025, 0.025] and ext.nbox >= 1
    assert env.root_state_tensor.shape == (3 * n, 13) and env.root_state_tensor.data_ptr() == sim.root_state.data_ptr()
    assert env.hand_indices.tolist() == list(range(0, 3 * n, 3)) and env.object_indices.tolist() == list(range(1, 3 * n, 3))
    assert env.rigid_body_states.shape[1] == sim.nb + 2 and len(env.fingertip_handles) == 5
    rs = sim.root_state.view(n, 3, 13)
    assert torch.allclose(rs[:, 0, 0:3], torch.tensor([0.0, 0.0, 0.5])) and torch.allclose(rs[:, 1, 0:3], torch.tensor([0.0, -0.39, 0.6]))
    torch.manual_seed(0)
    obs, rew, reset, extras = env.step(2 * torch.rand(n, 20) - 1)          # first step resets every env and every goal
    assert sim.steps == 1 and obs["obs"].shape == (n, 211) and torch.isfinite(obs["obs"]).all() and torch.isfinite(rew).all()
    lo, hi = env.shadow_hand_dof_lower_limits, env.shadow_hand_dof_upper_limits
    assert ((env.shadow_hand_dof_pos >= lo - 1e-6) & (env.shadow_hand_dof_pos <= hi + 1e-6)).all()
    # position targets reached the engine's tensor, clamped to the joint range (shadow_hand.py:684-698)
    assert ((sim.dof_target >= lo - 1e-6) & (sim.dof_target <= hi + 1e-6)).all() and sim.dof_target.abs().sum() > 0
    # reset_target_pose moved the goal marker's row; the cube was re-posed with noise
    assert (rs[:, 2, 3:7].norm(dim=-1) - 1).abs().max() < 1e-5 and (rs[:, 2, 3:7] - torch.tensor([0.0, 0, 0, 1])).abs().max() > 1e-3
    assert (rs[:, 1, 0:3] - torch.tensor([0.0, -0.39, 0.6])).abs().max() < 0.011
    assert "consecutive_successes" in extras and "time_outs" in extras


def test_procedural_primitive_assets_become_the_free_object(compat_cpu, reference_assets):
    """gym.create_sphere / create_box / create_capsule (ball_balance.py:277, franka_cube_stack.py:223-245): one primitive, mass =
    density x volume, and as the second actor of an env the engine's rounded box (sphere: a point + radius)."""
    from isaacgym import gymapi
    import math
    gym = gymapi.acquire_gym()
    sp = gymapi.SimParams(); sp.dt, sp.substeps = 0.01, 2
    sim = gym.create_sim(0, -1, gymapi.SIM_PHYSX, sp)
    gym.add_ground(sim, gymapi.PlaneParams())
    ao = gymapi.AssetOptions(); ao.density = 200.0
    ball = gym.create_sphere(sim, 0.1, ao)
    assert gym.get_asset_rigid_body_count(ball) == 1 and gym.get_asset_dof_count(ball) == 0
    assert abs(float(ball.model.mass[0]) - 200.0 * 4 / 3 * math.pi * 1e-3) < 1e-9
    box = gym.create_box(sim, 0.2, 0.4, 0.6, ao)
    assert abs(float(box.model.mass[0]) - 200.0 * 0.048) < 1e-9 and [round(float(v), 6) for v in box.model.geom_size[0]] == [0.1, 0.2, 0.3]
    cap = gym.create_capsule(sim, 0.05, 0.4, ao)
    assert abs(float(cap.model.mass[0]) - 200.0 * (math.pi * 0.05 ** 2 * 0.4 + 4 / 3 * math.pi * 0.05 ** 3)) < 1e-9
    # the ball as the free object of a two-actor env (articulation + ball): cartpole stands in for the articulation
    copt = gymapi.AssetOptions(); copt.fix_base_link = True; copt.angular_damping = 0.5
    cart = gym.load_asset(sim, reference_assets, "urdf/cartpole.urdf", copt)
    for i in range(2):
        e = gym.create_env(sim, gymapi.Vec3(-1, -1, 0), gymapi.Vec3(1, 1, 1), 2)
        gym.create_actor(e, cart, gymapi.Transform(gymapi.Vec3(0, 0, 2.0)), "cartpole", i, 1, 0)
        gym.create_actor(e, ball, gymapi.Transform(gymapi.Vec3(0.5, 0, 1.0)), "ball", i, 0, 0)
    gym.prepare_sim(sim)
    ext = sim.engine.ext
    assert ext.actors_per_env == 2 and ext.obj_actor == 1 and [float(v) for v in ext.obj_half] == [0.0, 0.0, 0.0]
    assert abs(ext.obj_round - 0.1) < 1e-7 and abs(ext.obj_mass - float(ball.model.mass[0])) < 1e-6 and ext.obj_max_angular_velocity == 64.0
    rs = sim.engine.root_state.view(2, 2, 13)
    assert torch.allclose(rs[:, 1, 0:3], torch.tensor([0.5, 0.0, 1.0]))


def test_name_maps_and_small_accessors_of_the_shim(compat_cpu, reference_assets):
    """the dictionary / count accessors other reference tasks use around the tensor API (franka_cube_stack.py:391, allegro_hand.py,
    ant.py:307-321 debug lines): body / DOF order = the tensors' order.  The scene is the one ant.py builds: one Ant per env."""
    from isaacgym import gymapi
    gym = gymapi.acquire_gym()
    sp = gymapi.SimParams(); sp.dt, sp.substeps = 0.0166, 2
    sim = gym.create_sim(0, -1, gymapi.SIM_PHYSX, sp)
    gym.add_ground(sim, gymapi.PlaneParams())
    ant = gym.load_asset(sim, reference_assets, "mjcf/nv_ant.xml", gymapi.AssetOptions())
    n = 4
    envs = []
    for i in range(n):
        envs.append(gym.create_env(sim, gymapi.Vec3(-2, -2, 0), gymapi.Vec3(2, 2, 2), 2))
        gym.create_actor(envs[i], ant, gymapi.Transform(gymapi.Vec3(0, 0, 0.44)), "ant", i, 1, 0)
    gym.prepare_sim(sim)
    e0 = envs[0]
    bd, dd = gym.get_actor_rigid_body_dict(e0, 0), gym.get_actor_dof_dict(e0, 0)
    assert len(bd) == 9 and len(dd) == 8 and bd["torso"] == 0 and sorted(dd.values()) == list(range(8))
    assert gym.get_actor_rigid_body_names(e0, 0)[bd["front_left_foot"]] == "front_left_foot"
    assert gym.find_actor_dof_handle(e0, 0, gym.get_actor_dof_names(e0, 0)[3]) == 3
    assert gym.get_sim_actor_count(sim) == n and gym.get_actor_dof_count(e0, 0) == 8 and gym.get_actor_rigid_body_count(e0, 0) == 9
    assert gym.get_asset_rigid_body_dict(sim.asset) == bd and gym.get_asset_dof_dict(sim.asset) == dd
    f = torch.arange(n * 8, dtype=torch.float32).view(n, 8)
    gym.set_dof_actuation_force_tensor_indexed(sim, f, torch.tensor([2, 0], dtype=torch.int32), 2)
    got = sim.engine.dof_actuation.view(n, 8)
    assert torch.equal(got[2], f[2]) and torch.equal(got[0], f[0]) and float(got[1].abs().sum()) == 0.0
    gym.add_lines(None, None, 0, [], []); gym.clear_lines(None); gym.debug_print_asset(sim.asset)


@needs_reference
def test_reference_shadow_hand_random_forces_reach_the_engine(compat_cpu):
    """env.forceScale > 0 (shadow_hand.py:700-709): the reference's own pre_physics_step calls
    apply_rigid_body_force_tensors(rb_forces, None, LOCAL_SPACE); the shim hands the object's row to the engine for
    exactly one simulate() and rejects forces it would silently drop."""
    import importlib
    from isaacgym import gymapi
    mod = importlib.import_module("isaacgymenvs.tasks.shadow_hand")
    n = 64
    cfg = _cfg("ShadowHand", n)
    cfg["env"]["forceScale"] = 2.0; cfg["env"]["forceProbRange"] = [0.5, 0.9]
    env = mod.ShadowHand(cfg=cfg, rl_device="cpu", sim_device="cpu", graphics_device_id=-1, headless=True,
                         virtual_screen_capture=False, force_render=False)
    sim = env.sim.engine
    torch.manual_seed(0)
    env.step(2 * torch.rand(n, 20) - 1)
    obj = int(env.object_rb_handles[0])
    assert obj == sim.nb                                                   # the object's body follows the hand's bodies
    drew = env.rb_forces[:, obj].abs().sum(-1) > 0
    assert 0.3 * n < int(drew.sum()) < n                                   # rand < prob with prob in [0.5, 0.9]
    assert torch.equal(sim.seen_obj_force, env.rb_forces[:, obj])          # what simulate() saw: the LOCAL_SPACE force, unchanged
    assert float(sim.tensors[sim.E.T_OBJ_FORCE].abs().max()) == 0.0       # cleared after the step, as PhysX clears applied forces
    gym = env.gym
    bad = torch.zeros_like(env.rb_forces); bad[:, 3, 0] = 1.0
    with pytest.raises(NotImplementedError):
        gym.apply_rigid_body_force_tensors(env.sim, bad, None, gymapi.LOCAL_SPACE)
    with pytest.raises(NotImplementedError):
        gym.apply_rigid_body_force_tensors(env.sim, None, bad, gymapi.LOCAL_SPACE)
    # ENV_SPACE forces are turned into the object's frame
    f = torch.zeros_like(env.rb_forces); f[:, obj, 2] = 1.0
    gym.apply_rigid_body_force_tensors(env.sim, f, None, gymapi.ENV_SPACE)
    from isaacgymenvs.utils.torch_jit_utils import quat_rotate_inverse
    q = sim.root_state.view(n, 3, 13)[:, 1, 3:7]
    assert torch.allclose(sim.tensors[sim.E.T_OBJ_FORCE], quat_rotate_inverse(q, f[:, obj]), atol=1e-6)


@needs_reference
@pytest.mark.parametrize("obj,half,rnd,mass", [("pen", [0.0, 0.0, 0.1], 0.008, 0.042357), ("egg", [0.0, 0.0, 0.01], 0.03, 0.150796)])
def test_reference_shadow_hand_egg_and_pen_reach_the_engine_as_rounded_boxes(compat_cpu, obj, half, rnd, mass):
    """env.objectType egg / pen (shadow_hand.py:84-99): the reference loads egg.xml / pen.xml itself; the shim turns the single
    collision primitive into the engine's rounded box and passes the object's own AssetOptions (speed limit 64 rad/s, damping)."""
    import importlib
    mod = importlib.import_module("isaacgymenvs.tasks.shadow_hand")
    cfg = _cfg("ShadowHand", 4)
    cfg["env"]["objectType"] = obj
    env = mod.ShadowHand(cfg=cfg, rl_device="cpu", sim_device="cpu", graphics_device_id=-1, headless=True,
                         virtual_screen_capture=False, force_render=False)
    ext = env.sim.engine.ext
    assert ext.actors_per_env == 3 and ext.obj_actor == 1
    assert [round(float(v), 6) for v in ext.obj_half] == half and abs(ext.obj_round - rnd) < 1e-7 and abs(ext.obj_mass - mass) < 1e-5
    assert ext.obj_max_angular_velocity == 64.0 and abs(ext.obj_angular_damping - 0.5) < 1e-7
    assert env.ignore_z == (obj == "pen")
    obs, rew, reset, extras = env.step(torch.zeros(4, 20))
    assert torch.isfinite(obs["obs"]).all()


@needs_reference
def test_unmodified_reference_flat_anymal_runs_on_the_shim(compat_cpu):
    """SURVEY 8f rank 2: tasks/anymal.py drives PhysX position drives (DOF_MODE_POS via set_actor_dof_properties,
    set_dof_position_target_tensor) and reads net contact forces -- unmodified on the shim."""
    import importlib
    mod = importlib.import_module("isaacgymenvs.tasks.anymal")
    assert os.path.realpath(mod.__file__).startswith(REFERENCE)
    n = 8
    env = mod.Anymal(cfg=_cfg("Anymal", n), rl_device="cpu", sim_device="cpu", graphics_device_id=-1, headless=True,
                     virtual_screen_capture=False, force_render=False)
    sim = env.sim.engine
    assert env.num_obs == 48 and env.num_acts == 12
    m = sim.model
    assert (m.drive_mode[1:] == 1).all() and np.allclose(m.kp[1:], 85.0) and np.allclose(m.kd[1:], 2.0)     # anymal.py:199-203
    obs, rew, reset, extras = env.step(2 * torch.rand(n, 12) - 1)
    assert obs["obs"].shape == (n, 48) and torch.isfinite(obs["obs"]).all() and torch.isfinite(rew).all()
    # targets = action_scale * actions + default_dof_pos reached the engine's target tensor (anymal.py:226-229)
    assert torch.allclose(sim.dof_target, 0.5 * env.actions + env.default_dof_pos)


@needs_reference
def test_unmodified_reference_anymal_terrain_runs_on_the_shim(compat_cpu):
    """tasks/anymal_terrain.py builds its terrain with isaacgym.terrain_utils (restated in isaacgymenvs_b200/terrain.py),
    converts it to a triangle mesh and calls gym.add_triangle_mesh; the shim hands the engine the underlying height field."""
    import importlib
    mod = importlib.import_module("isaacgymenvs.tasks.anymal_terrain")
    assert os.path.realpath(mod.__file__).startswith(REFERENCE)
    n = 16
    cfg = _cfg("AnymalTerrain", n)
    cfg["env"]["terrain"]["numLevels"] = 2; cfg["env"]["terrain"]["numTerrains"] = 2
    env = mod.AnymalTerrain(cfg=cfg, rl_device="cpu", sim_device="cpu", graphics_device_id=-1, headless=True,
                            virtual_screen_capture=False, force_render=False)
    sim = env.sim.engine
    assert env.num_obs == 188 and env.num_acts == 12
    t = env.terrain
    assert np.array_equal(sim.kw["hfield"], t.height_field_raw) and sim.kw["hfield"].dtype == np.int16
    assert sim.kw["hf_horizontal_scale"] == t.horizontal_scale and sim.kw["hf_vertical_scale"] == t.vertical_scale
    assert sim.kw["hf_origin"] == (-t.border_size, -t.border_size)
    assert t.vertices.shape == (t.tot_rows * t.tot_cols, 3) and t.triangles.shape == (2 * (t.tot_rows - 1) * (t.tot_cols - 1), 3)
    # the mesh follows the samples: every vertex height is its sample's
    assert np.allclose(np.asarray(t.vertices)[:, 2].reshape(t.tot_rows, t.tot_cols), t.height_field_raw * t.vertical_scale)
    obs, rew, reset, extras = env.step(2 * torch.rand(n, 12) - 1)
    assert sim.steps == env.decimation + env.control_freq_inv and obs["obs"].shape == (n, 188) and torch.isfinite(obs["obs"]).all()
    assert torch.isfinite(rew).all() and "time_outs" in extras
