"""Golden vectors for ShadowHand from the REFERENCE's own code (build container only):
    python tests/golden/make_golden_hand.py
`tasks/shadow_hand.py` is loaded by path with isaacgym stubbed; an instance is made without running __init__ and its
METHODS pre_physics_step (:661-705, which calls reset_target_pose :594-610 and reset_idx :612-659), post_physics_step
(:707-712), compute_observations (:436-458 -> the four layouts :460-592) and compute_reward (:415-424 ->
compute_hand_reward :749-804) run unmodified on CPU torch.  Two things are injected, both outside the reference's
arithmetic: `torch_rand_float` returns the engine's counter-based Philox numbers (so resets are reproducible per env),
and the closed `gym.refresh_rigid_body_state_tensor` is played by the oracle's forward kinematics.
Output: tests/golden/shadow_hand.npz."""
import importlib.util
import os
import sys
import types
import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
REF = "/root/reference/isaacgymenvs"
OUT = os.path.dirname(os.path.abspath(__file__))
SEED = 42


def load():
    for name in ("isaacgym", "isaacgym.gymtorch", "isaacgym.gymapi", "isaacgym.gymutil", "isaacgym.terrain_utils"):
        sys.modules.setdefault(name, types.ModuleType(name))
    sys.modules["isaacgym"].gymtorch = sys.modules["isaacgym.gymtorch"]
    sys.modules["isaacgym"].gymapi = sys.modules["isaacgym.gymapi"]
    sys.modules["isaacgym"].gymutil = sys.modules["isaacgym.gymutil"]
    sys.modules["isaacgym.gymtorch"].unwrap_tensor = lambda t: t
    sys.modules["isaacgym.gymapi"].LOCAL_SPACE = 1              # only named in the apply_rigid_body_force_tensors call (:708)
    for name in ("isaacgymenvs", "isaacgymenvs.utils", "isaacgymenvs.tasks", "isaacgymenvs.tasks.base"):
        sys.modules.setdefault(name, types.ModuleType(name))
    sys.modules["isaacgymenvs.tasks"].__path__ = []
    vt = types.ModuleType("isaacgymenvs.tasks.base.vec_task"); vt.VecTask = type("VecTask", (), {})
    sys.modules["isaacgymenvs.tasks.base.vec_task"] = vt

    def ld(modname, rel):
        spec = importlib.util.spec_from_file_location(modname, os.path.join(REF, rel))
        mod = importlib.util.module_from_spec(spec); sys.modules[modname] = mod; spec.loader.exec_module(mod)
        return mod
    tju = ld("isaacgymenvs.utils.torch_jit_utils", "utils/torch_jit_utils.py")
    sh = ld("isaacgymenvs.tasks.shadow_hand", "tasks/shadow_hand.py")
    return tju, sh


class Gym:
    """The closed gym.* calls the methods make: setters are no-ops (the tensors ARE the state), refresh of the rigid-body
    tensor is forward kinematics by the oracle."""

    def __init__(self, task, orc, model):
        self.t, self.orc, self.m = task, orc, model

    def __getattr__(self, name):
        if name == "refresh_rigid_body_state_tensor":
            return self._fk
        return lambda *a, **k: None

    def _fk(self, sim):
        t, m = self.t, self.m
        n = t.num_envs
        root = t.root_state_tensor.view(n, 3, 13)[:, 0].numpy().astype(np.float64)
        dof = t.dof_state.view(n, -1, 2).numpy().astype(np.float64)
        bs = self.orc.body_states(np.ascontiguousarray(root), np.ascontiguousarray(dof)).astype(np.float32)
        full = np.concatenate([bs, t.root_state_tensor.view(n, 3, 13)[:, 1:3].numpy()], 1)
        t.rigid_body_states = torch.tensor(full)


def make_case(sh, g, n, obs_type, relative, mcs, mavg, fall_penalty, orc, model, act_idx, fingertip_handles, force=None, object_type="block"):
    """force: None, or dict(scale, prob_range, obj_mass) -- random forces on the object (shadow_hand.py:700-709); the
    reference's torch.rand / torch.randn draws are then played by the engine's counter-based stream as well."""
    from oracle import tasks_np
    D = model.ndof
    t = object.__new__(sh.ShadowHand)
    t.num_envs, t.device, t.randomize, t.num_shadow_hand_dofs, t.num_actions = n, "cpu", False, D, 20
    t.up_axis_idx, t.object_type, t.obs_type, t.asymmetric_obs = 2, object_type, obs_type, False
    t.num_fingertips, t.viewer, t.debug_viz, t.print_success_stat = 5, None, False, False
    t.sim = None
    lo = torch.tensor(model.lower[1:], dtype=torch.float); hi = torch.tensor(model.upper[1:], dtype=torch.float)
    t.shadow_hand_dof_lower_limits, t.shadow_hand_dof_upper_limits = lo, hi
    t.shadow_hand_dof_default_pos = torch.zeros(D); t.shadow_hand_dof_default_vel = torch.zeros(D)
    t.shadow_hand_default_dof_pos = torch.zeros(D)
    t.actuated_dof_indices = torch.tensor(act_idx, dtype=torch.long)
    t.fingertip_handles = torch.tensor(fingertip_handles, dtype=torch.long)
    t.x_unit_tensor = torch.tensor([1.0, 0, 0]).repeat(n, 1); t.y_unit_tensor = torch.tensor([0.0, 1, 0]).repeat(n, 1)
    t.z_unit_tensor = torch.tensor([0.0, 0, 1]).repeat(n, 1)
    t.reset_position_noise, t.reset_dof_pos_noise, t.reset_dof_vel_noise = 0.01, 0.2, 0.05
    t.force_scale, t.force_decay, t.force_decay_interval = 0.0, torch.tensor(0.99), 0.08
    t.force_prob_range = torch.tensor([0.001, 0.1]); t.random_force_prob = torch.zeros(n)
    t.rb_forces = torch.zeros(n, model.nb + 2, 3)
    t.use_relative_control, t.shadow_hand_dof_speed_scale, t.dt, t.act_moving_average = relative, 20.0, 0.01667, mavg
    t.max_episode_length, t.dist_reward_scale, t.rot_reward_scale, t.rot_eps = 600, -10.0, 1.0, 0.1
    t.action_penalty_scale, t.success_tolerance, t.reach_goal_bonus, t.fall_dist, t.fall_penalty = -0.0002, 0.1, 250, 0.24, fall_penalty
    t.max_consecutive_successes, t.av_factor = mcs, torch.tensor(0.1)
    t.vel_obs_scale, t.force_torque_obs_scale = 0.2, 10.0
    t.extras = {}
    # ---- state
    hand_q = torch.tensor(np.asarray(model.default_root_quat), dtype=torch.float)
    rs = torch.zeros(n, 3, 13); rs[:, :, 6] = 1
    rs[:, 0, 0:3] = torch.tensor([0.0, 0.0, 0.5]); rs[:, 0, 3:7] = hand_q
    obj_init = torch.zeros(n, 13); obj_init[:, 0:3] = torch.tensor([0.0, -0.39, 0.6]); obj_init[:, 6] = 1
    t.object_init_state = obj_init
    goal_init = obj_init.clone(); goal_init[:, 2] -= 0.04
    t.goal_init_state = goal_init
    t.goal_displacement_tensor = torch.tensor([-0.2, -0.06, 0.12])
    gq = torch.randn(n, 4, generator=g); gq /= gq.norm(dim=-1, keepdim=True)
    t.goal_states = goal_init.clone(); t.goal_states[:, 3:7] = gq
    # object: a third near the goal pose (successes), a third far (falls), the rest in between
    oq = torch.randn(n, 4, generator=g); oq /= oq.norm(dim=-1, keepdim=True)
    k = n // 3
    small = torch.randn(k, 4, generator=g) * 0.03; small[:, 3] = 1.0
    small /= small.norm(dim=-1, keepdim=True)
    tju = sys.modules["isaacgymenvs.utils.torch_jit_utils"]
    oq[:k] = tju.quat_mul(small, gq[:k])
    rs[:, 1, 0:3] = goal_init[:, 0:3] + torch.randn(n, 3, generator=g) * 0.05
    rs[k:2 * k, 1, 0:3] += torch.tensor([0.0, 0.0, -0.3])
    rs[:, 1, 3:7] = oq
    rs[:, 1, 7:13] = torch.randn(n, 6, generator=g)
    rs[:, 2, 0:3] = t.goal_states[:, 0:3] + t.goal_displacement_tensor; rs[:, 2, 3:7] = gq
    t.root_state_tensor = rs.view(3 * n, 13).clone()
    t.hand_indices = torch.arange(0, 3 * n, 3); t.object_indices = t.hand_indices + 1; t.goal_object_indices = t.hand_indices + 2
    u = torch.rand(n, D, generator=g) * 1.1 - 0.05
    t.dof_state = torch.stack([lo + (hi - lo) * u, torch.randn(n, D, generator=g) * 2.0], -1).view(n * D, 2).contiguous()
    t.shadow_hand_dof_state = t.dof_state.view(n, -1, 2)[:, :D]
    t.shadow_hand_dof_pos = t.shadow_hand_dof_state[..., 0]; t.shadow_hand_dof_vel = t.shadow_hand_dof_state[..., 1]
    t.prev_targets = lo + (hi - lo) * torch.rand(n, D, generator=g)
    t.cur_targets = t.prev_targets.clone()
    t.vec_sensor_tensor = torch.randn(n, 30, generator=g); t.dof_force_tensor = torch.randn(n, D, generator=g) * 0.3
    t.reset_buf = (torch.rand(n, generator=g) < 0.2).long()
    t.reset_goal_buf = (torch.rand(n, generator=g) < 0.2).long()
    t.progress_buf = torch.randint(0, 602, (n,), generator=g)
    t.randomize_buf = torch.zeros(n, dtype=torch.long)
    t.successes = torch.randint(0, 60, (n,), generator=g).float()
    t.consecutive_successes = torch.tensor([3.25])
    t.rew_buf = torch.zeros(n); t.obs_buf = torch.zeros(n, {"openai": 42, "full_no_vel": 77, "full": 157, "full_state": 211}[obs_type])
    reset_count = torch.randint(0, 5, (n,), generator=g).int(); goal_count = torch.randint(0, 5, (n,), generator=g).int()
    actions = torch.rand(n, 20, generator=g) * 2.4 - 1.2
    t.gym = Gym(t, orc, model)
    force_in = {}
    if force is not None:
        t.force_scale = force["scale"]
        t.force_prob_range = torch.tensor(force["prob_range"], dtype=torch.float)
        t.random_force_prob = torch.rand(n, generator=g) * 0.6
        t.object_rb_handles = torch.tensor([model.nb], dtype=torch.long)
        t.object_rb_masses = torch.tensor([force["obj_mass"]], dtype=torch.float)
        t.rb_forces[:, model.nb] = torch.randn(n, 3, generator=g) * 0.05
        force_in = dict(obj_force=t.rb_forces[:, model.nb].numpy().copy(), force_prob=t.random_force_prob.numpy().copy())
    inputs = dict(root=t.root_state_tensor.numpy().copy(), dof_state=t.dof_state.numpy().copy(), prev_targets=t.prev_targets.numpy().copy(),
                  cur_targets=t.cur_targets.numpy().copy(), goal_states=t.goal_states.numpy().copy(), sensors=t.vec_sensor_tensor.numpy().copy(),
                  dof_force=t.dof_force_tensor.numpy().copy(), reset=t.reset_buf.numpy().copy(), reset_goal=t.reset_goal_buf.numpy().copy(),
                  progress=t.progress_buf.numpy().copy(), successes=t.successes.numpy().copy(), cons=t.consecutive_successes.numpy().copy(),
                  reset_count=reset_count.numpy().copy(), goal_reset_count=goal_count.numpy().copy(), actions=actions.numpy().copy(),
                  object_init=obj_init.numpy().copy(), goal_init=goal_init.numpy().copy(), **force_in)

    # ---- the engine's Philox numbers behind torch_rand_float
    ctx = {"env_ids": None, "in_reset_idx": False}
    orig_rtp, orig_ri = sh.ShadowHand.reset_target_pose, sh.ShadowHand.reset_idx

    def rand_float(lower, upper, shape, device):
        ids = ctx["env_ids"].tolist()
        assert lower == -1.0 and upper == 1.0 and shape[0] == len(ids)
        rows = []
        for e in ids:
            if ctx["in_reset_idx"]:
                r = tasks_np.hand_rand_floats(SEED, e, int(reset_count[e]), 2 * D + 7)
                rows.append(r[:2 * D + 5] if shape[1] == 2 * D + 5 else np.concatenate([r[2 * D + 5:2 * D + 7], np.zeros(2, np.float32)]))
            else:
                gcount = (int(goal_count[e]) | 0x80000000) & 0xFFFFFFFF
                rows.append(np.concatenate([tasks_np.hand_rand_floats(SEED, e, gcount, 2), np.zeros(2, np.float32)]))
        return torch.tensor(np.stack(rows).astype(np.float32)) if rows else torch.zeros(shape)

    def rtp(self, env_ids, apply_reset=False):
        ctx["env_ids"] = env_ids
        return orig_rtp(self, env_ids, apply_reset)

    def ri(self, env_ids, goal_env_ids):
        ctx["env_ids"] = env_ids; ctx["in_reset_idx"] = True
        try:
            return orig_ri(self, env_ids, goal_env_ids)
        finally:
            ctx["in_reset_idx"] = False
    # torch.rand / torch.randn of the force block (:704-706) and of reset_idx's random_force_prob (:642), when forces are on
    class TorchProxy:
        def __getattr__(self, name):
            return getattr(torch, name)

        def rand(self, k, device=None):
            if ctx["in_reset_idx"]:                            # one uniform per env of env_ids: index 2 D + 7 of its reset stream
                ids = ctx["env_ids"].tolist(); assert k == len(ids)
                return torch.tensor([float(tasks_np.reset_uniforms(SEED, e, int(reset_count[e]), 2 * D + 8)[2 * D + 7]) for e in ids], dtype=torch.float)
            assert k == n                                       # the force block: one uniform per env, step = progress, count after resets
            cnt = reset_count.clone(); cnt[inputs["reset"] != 0] += 1
            dr = [tasks_np.hand_force_draws(SEED, e, int(cnt[e]), int(t.progress_buf[e])) for e in range(n)]
            ctx["normals"] = np.stack([d[1] for d in dr])
            return torch.tensor(np.array([d[0] for d in dr], np.float32))

        def randn(self, shape, device=None):
            # rows of the envs that drew a new force, in order: what `(rand < prob).nonzero()` selected
            hit = (torch.tensor(ctx["u_last"]) < t.random_force_prob).nonzero().flatten().tolist()
            assert tuple(shape) == (len(hit), 1, 3)
            return torch.tensor(ctx["normals"][hit].reshape(len(hit), 1, 3))
    proxy = TorchProxy()
    _rand = proxy.rand

    def rand_keep(k, device=None):
        r = _rand(k, device)
        if not ctx["in_reset_idx"]:
            ctx["u_last"] = r.numpy().copy()
        return r
    proxy.rand = rand_keep
    sh.torch_rand_float = rand_float
    sh.ShadowHand.reset_target_pose, sh.ShadowHand.reset_idx = rtp, ri
    if force is not None:
        sh.torch = proxy
    try:
        a = torch.clamp(actions, -1.0, 1.0)                    # VecTask.step, vec_task.py:374
        t.pre_physics_step(a)
        t.post_physics_step()                                   # control_freq_inv == 0: no simulate in between
    finally:
        sh.ShadowHand.reset_target_pose, sh.ShadowHand.reset_idx = orig_rtp, orig_ri
        sh.torch = torch
    timeout = (t.progress_buf >= t.max_episode_length - 1) & (t.reset_buf != 0)                     # vec_task.py:394
    outputs = dict(root=t.root_state_tensor.numpy(), dof_state=t.dof_state.numpy(), prev_targets=t.prev_targets.numpy(),
                   cur_targets=t.cur_targets.numpy(), goal_states=t.goal_states.numpy(), obs=t.obs_buf.numpy(), rew=t.rew_buf.numpy(),
                   reset=t.reset_buf.numpy(), reset_goal=t.reset_goal_buf.numpy(), progress=t.progress_buf.numpy(),
                   successes=t.successes.numpy(), cons=t.consecutive_successes.numpy(), timeout=timeout.numpy(),
                   fingertip_state=t.fingertip_state.numpy())
    if force is not None:
        others = t.rb_forces.clone(); others[:, model.nb] = 0
        outputs.update(obj_force=t.rb_forces[:, model.nb].numpy().copy(), force_prob=t.random_force_prob.numpy().copy(),
                       other_forces=np.float32(others.abs().sum()))
    return inputs, outputs


def main():
    from tests.hand_common import hand_setup, DT, SUBSTEPS, G
    from oracle.oracle import OracleSim
    tju, sh = load()
    model, obj, tendons = hand_setup()
    orc = OracleSim(model, DT, SUBSTEPS, G, obj=obj, tendons=tendons, tendon_k=30.0, tendon_d=0.1)
    names = list(model.dof_names)
    act_idx = [names.index(j) for j in model.actuator_joint]
    ft = [int(b) for b in model.sensor_body]
    n = 120                 # keeps the file under 1 MB while every case still resets more than 10 envs and 10 goals
    blob = {"seed": np.int64(SEED), "actuated": np.array(act_idx, np.int32), "fingertips": np.array(ft, np.int32)}
    cases = {"a": dict(relative=False, mcs=0, mavg=1.0, fall_penalty=0.0), "b": dict(relative=True, mcs=50, mavg=1.0, fall_penalty=-50.0),
             "c": dict(relative=False, mcs=0, mavg=0.3, fall_penalty=0.0)}
    for cname, kw in cases.items():
        for obs_type in ("full_state", "full", "full_no_vel", "openai"):
            if cname != "a" and obs_type != "full_state":
                continue
            g = torch.Generator().manual_seed({"a": 11, "b": 12, "c": 13}[cname])
            inp, out = make_case(sh, g, n, obs_type, orc=orc, model=model, act_idx=act_idx, fingertip_handles=ft, **kw)
            if obs_type == "full_state":
                for k, v in inp.items():
                    blob[f"{cname}_in_{k}"] = v
                for k, v in out.items():
                    blob[f"{cname}_out_{k}"] = v
            else:
                blob[f"{cname}_out_obs_{obs_type}"] = out["obs"]
    np.savez_compressed(os.path.join(OUT, "shadow_hand.npz"), **blob)
    print("wrote shadow_hand.npz;", {k: v.shape for k, v in blob.items() if k.startswith("a_out")})


def main_force():
    """Case "f": forceScale 2.0, forceProbRange [0.05, 0.5] -> tests/golden/shadow_hand_force.npz (separate file: the
    fixtures of main() stay byte-identical)."""
    from tests.hand_common import hand_setup, DT, SUBSTEPS, G
    from oracle.oracle import OracleSim
    tju, sh = load()
    model, obj, tendons = hand_setup()
    orc = OracleSim(model, DT, SUBSTEPS, G, obj=obj, tendons=tendons, tendon_k=30.0, tendon_d=0.1)
    names = list(model.dof_names)
    act_idx = [names.index(j) for j in model.actuator_joint]
    ft = [int(b) for b in model.sensor_body]
    g = torch.Generator().manual_seed(14)
    force = dict(scale=2.0, prob_range=[0.05, 0.5], obj_mass=float(obj["mass"]))
    inp, out = make_case(sh, g, 256, "full_state", relative=False, mcs=0, mavg=1.0, fall_penalty=0.0, orc=orc, model=model,
                         act_idx=act_idx, fingertip_handles=ft, force=force)
    blob = {"seed": np.int64(SEED), "actuated": np.array(act_idx, np.int32), "fingertips": np.array(ft, np.int32),
            "force_scale": np.float32(force["scale"]), "force_prob_range": np.array(force["prob_range"], np.float32),
            "obj_mass": np.float32(force["obj_mass"])}
    for k, v in inp.items():
        blob[f"f_in_{k}"] = v
    for k, v in out.items():
        blob[f"f_out_{k}"] = v
    np.savez_compressed(os.path.join(OUT, "shadow_hand_force.npz"), **blob)
    print("wrote shadow_hand_force.npz; new forces drawn in", int((out["obj_force"] != inp["obj_force"] * np.float32(0.99 ** (0.01667 / 0.08))).any(1).sum()), "of 256 envs")


def main_pen():
    """Case "p": objectType pen -- reset_idx poses the object with randomize_rotation_pen (:626-629) and compute_reward passes
    ignore_z_rot (:421, :758-759: twice the success tolerance) -> tests/golden/shadow_hand_pen.npz (128 envs)."""
    from tests.hand_common import hand_setup, DT, SUBSTEPS, G
    from oracle.oracle import OracleSim
    tju, sh = load()
    model, obj, tendons = hand_setup()
    orc = OracleSim(model, DT, SUBSTEPS, G, obj=obj, tendons=tendons, tendon_k=30.0, tendon_d=0.1)
    names = list(model.dof_names)
    act_idx = [names.index(j) for j in model.actuator_joint]
    ft = [int(b) for b in model.sensor_body]
    g = torch.Generator().manual_seed(15)
    inp, out = make_case(sh, g, 128, "full_state", relative=False, mcs=0, mavg=1.0, fall_penalty=0.0, orc=orc, model=model,
                         act_idx=act_idx, fingertip_handles=ft, object_type="pen")
    blob = {"seed": np.int64(SEED), "actuated": np.array(act_idx, np.int32), "fingertips": np.array(ft, np.int32)}
    for k, v in inp.items():
        blob[f"p_in_{k}"] = v
    for k, v in out.items():
        blob[f"p_out_{k}"] = v
    np.savez_compressed(os.path.join(OUT, "shadow_hand_pen.npz"), **blob)
    print("wrote shadow_hand_pen.npz; resets", int(inp["reset"].sum()), "successes counted", int((out["successes"] - inp["successes"] * (inp["reset"] == 0)).sum()))


if __name__ == "__main__":
    if "--pen" in sys.argv:
        main_pen()
    elif "--force" in sys.argv:
        main_force()
    else:
        main()
