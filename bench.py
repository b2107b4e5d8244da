#!/usr/bin/env python
"""bench.py -- env-steps/s of the fused VecTask.step() hot path (BASELINE.json metric).

    python bench.py --gpus 1 --steps 200 --warmup 5            # Ant, num_envs=16384 per GPU
    torchrun --nproc-per-node N ... bench.py --gpus N ...       # weak scaling: 16384 envs per rank (--scaling strong: 16384 in total)
    python bench.py --impl reference ...                        # CPU port of the path (oracle/), host cores, same config
    python bench.py --workload humanoid|anymal|shadow_hand|cartpole
    python bench.py ... --dump-outputs DIR                      # also write what the last timed step returned, DIR/<name>.npy

One "step" = one VecTask.step() over all envs under random actions U(-1,1) (the README rollout loop of the reference,
README.md:39-51).  `value` is measured THROUGH `env.step(actions)` (the reference's metric, tasks/base/vec_task.py:360-408);
`device_only` times the same steps as bare C-ABI launches (what the roofline fraction is computed from).
Prints ONE JSON line on rank 0.
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

WORKLOADS = {   # name -> (task, num_envs per GPU, algorithmic bytes per env-step: SURVEY.md 8d / DESIGN.md)
    "ant": ("Ant", 16384, 673),
    "humanoid": ("Humanoid", 8192, 1161),
    "cartpole": ("Cartpole", 16384, 89),
    "anymal": ("AnymalTerrain", 4096, 2250),
    "shadow_hand": ("ShadowHand", 4096, 3640),    # BASELINE.json config 5: 32768 envs over 8 GPUs
}
METRIC = "env-steps/s at num_envs=16384 (Ant), 1/2/4/8 B200; %HBM roofline"
PARITY_NOTE = ("obs/reward/reset arithmetic pinned by the reference's own functions; physics parity UNPINNED against PhysX "
               "(closed gym.simulate): engine == own fp64 oracle only")


def measured_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured"
    except Exception:
        return 6650.0, "fallback"


class ClockSampler:
    """nvidia-smi clocks + throttle reasons during the timed region (B200_PROFILING.md)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx = float(r[1])
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


def make_env(task, n, device, rank):
    import isaacgymenvs_b200
    from isaacgymenvs_b200 import config
    cfg = config.builtin_cfg(task, {"sim_device": device, "rl_device": device})
    cfg["task"]["env_id_offset"] = rank * n
    return isaacgymenvs_b200.make(seed=42, task=task, num_envs=n, sim_device=device, rl_device=device,
                                  headless=True, cfg=cfg)


# ------------------------------------------------------------------------------------ CPU legs
def _loco_cpu(task, n_envs, threads):
    """Ant / Humanoid control step on host cores: oracle physics (C, float32, pthreads over envs) + the numpy
    restatement of the reference's obs/reward functions.  Returns the step closure."""
    import copy
    from isaacgymenvs_b200.assets import load_compiled
    from isaacgymenvs_b200 import config
    from oracle.oracle import OracleSim
    from oracle import tasks_np as T
    f32 = np.float32
    hum = task == "Humanoid"
    e = config.builtin_cfg(task, {})["task"]["env"]
    m = copy.deepcopy(load_compiled("humanoid" if hum else "ant"))
    if hum:
        m.sensor_body = np.array([m.body_names.index("right_foot"), m.body_names.index("left_foot")], dtype=np.int32)
    else:
        m.sensor_body = np.array([i for i, nme in enumerate(m.body_names) if "foot" in nme], dtype=np.int32)
    ns = len(m.sensor_body)
    m.sensor_pos = np.zeros((ns, 3)); m.sensor_quat = np.tile([0, 0, 0, 1.0], (ns, 1))
    nd = m.ndof
    sim = OracleSim(m, 0.0166, 2, precision="f32", threads=threads)
    rng = np.random.default_rng(42)
    gears = np.asarray(m.actuator_gear, f32)
    lo = np.minimum(m.lower[1:], m.upper[1:]).astype(f32); hi = np.maximum(m.lower[1:], m.upper[1:]).astype(f32)
    init = np.where(lo > 0, lo, np.where(hi < 0, hi, 0)).astype(f32)
    z0 = f32(1.34 if hum else 0.44)
    root = np.zeros((n_envs, 13), f32); root[:, 2] = z0; root[:, 6] = 1
    dof = np.zeros((n_envs, nd, 2), f32); dof[..., 0] = init
    st = dict(pot=np.full(n_envs, -1000.0 / 0.0166, f32), progress=np.zeros(n_envs, np.int64), reset=np.zeros(n_envs, np.int64))
    targets = np.tile(f32([1000, 0, 0]), (n_envs, 1)); isr = np.tile(f32([0, 0, 0, 1]), (n_envs, 1))
    b0 = np.tile(f32([1, 0, 0]), (n_envs, 1)); b1 = np.tile(f32([0, 0, 1]), (n_envs, 1))

    def one():
        a = np.clip(rng.uniform(-1, 1, size=(n_envs, nd)).astype(f32), -1, 1)
        out = sim.simulate(root, dof, a * gears[None] * f32(e["powerScale"]))
        st["progress"] += 1
        ids = np.nonzero(st["reset"])[0]
        if len(ids):
            dof[ids, :, 0] = np.clip(init + rng.uniform(-0.2, 0.2, size=(len(ids), nd)).astype(f32), lo, hi)
            dof[ids, :, 1] = rng.uniform(-0.1, 0.1, size=(len(ids), nd)).astype(f32)
            root[ids] = 0; root[ids, 2] = z0; root[ids, 6] = 1
            st["pot"][ids] = T.potentials_from(targets[ids] - root[ids, :3], 0.0166)
            st["progress"][ids] = 0
        zeros = np.zeros(n_envs, np.int64)
        if hum:
            obs, pot2, prev, _, _ = T.humanoid_observations(root, targets, st["pot"], isr, dof[..., 0], dof[..., 1], out["dof_force"].astype(f32), lo, hi,
                                                            e["dofVelocityScale"], out["sensor"].reshape(n_envs, -1).astype(f32), a, 0.0166,
                                                            e["contactForceScale"], e.get("angularVelocityScale", 0.1), b0, b1)
            rew, st["reset"] = T.humanoid_reward(obs, zeros, st["progress"], a, e["upWeight"], e["headingWeight"], pot2, prev, e["actionsCost"],
                                                 e["energyCost"], e["jointsAtLimitCost"], float(gears.max()), gears, e["terminationHeight"],
                                                 e["deathCost"], float(e["episodeLength"]))
        else:
            obs, pot2, prev, _, _ = T.ant_observations(root, targets, st["pot"], isr, dof[..., 0], dof[..., 1], lo, hi, e["dofVelocityScale"],
                                                       out["sensor"].reshape(n_envs, -1).astype(f32), a, 0.0166, e["contactForceScale"], b0, b1)
            rew, st["reset"] = T.ant_reward(obs, zeros, st["progress"], a, e["upWeight"], e["headingWeight"], pot2, prev, e["actionsCost"],
                                            e["energyCost"], e["jointsAtLimitCost"], e["terminationHeight"], e["deathCost"], float(e["episodeLength"]))
        st["pot"] = pot2
    return one


def _cartpole_cpu(n_envs, threads):
    import copy
    from isaacgymenvs_b200.assets import load_compiled
    from oracle.oracle import OracleSim
    from oracle import tasks_np as T
    f32 = np.float32
    m = copy.deepcopy(load_compiled("cartpole"))
    m.sensor_body = np.zeros(0, np.int32); m.sensor_pos = np.zeros((0, 3)); m.sensor_quat = np.zeros((0, 4))
    sim = OracleSim(m, 0.0166, 2, precision="f32", threads=threads)
    rng = np.random.default_rng(42)
    root = np.zeros((n_envs, 13), f32); root[:, 6] = 1; root[:, 2] = 2.0
    dof = np.zeros((n_envs, 2, 2), f32)
    st = dict(progress=np.zeros(n_envs, np.int64), reset=np.zeros(n_envs, np.int64))

    def one():
        a = np.clip(rng.uniform(-1, 1, size=(n_envs, 1)).astype(f32), -1, 1)
        tau = np.zeros((n_envs, 2), f32); tau[:, 0] = a[:, 0] * f32(400.0)
        sim.simulate(root, dof, tau)
        st["progress"] += 1
        ids = np.nonzero(st["reset"])[0]
        if len(ids):
            dof[ids, :, 0] = f32(0.2) * (rng.uniform(size=(len(ids), 2)).astype(f32) - f32(0.5))
            dof[ids, :, 1] = f32(0.5) * (rng.uniform(size=(len(ids), 2)).astype(f32) - f32(0.5))
            st["progress"][ids] = 0
        _, st["reset"] = T.cartpole_reward(dof[:, 1, 0], dof[:, 1, 1], dof[:, 0, 1], dof[:, 0, 0], 3.0, np.zeros(n_envs, np.int64), st["progress"], 500.0)
    return one


def _anymal_cpu(n_envs, threads):
    """AnymalTerrain control step on host cores: PD loop + 4+1 oracle simulates on the curriculum height field, then the
    numpy restatement of the reference's post_physics_step (prepare, termination, 13 reward terms, heights, 188-d obs).
    Resets re-spawn the robot on its tile without moving it through the terrain curriculum."""
    import copy
    from isaacgymenvs_b200.assets import load_compiled
    from isaacgymenvs_b200 import config
    from isaacgymenvs_b200.terrain import Terrain
    from oracle.oracle import OracleSim
    from oracle import tasks_np as T
    f32 = np.float32
    cfg = config.builtin_cfg("AnymalTerrain", {})["task"]
    e, learn = cfg["env"], cfg["env"]["learn"]
    m = copy.deepcopy(load_compiled("anymal"))
    m.sensor_body = np.zeros(0, np.int32); m.sensor_pos = np.zeros((0, 3)); m.sensor_quat = np.zeros((0, 4))
    ter = Terrain(e["terrain"], num_robots=n_envs, seed=42)
    hs = np.asarray(ter.heightsamples).reshape(ter.tot_rows, ter.tot_cols)
    sim = OracleSim(m, cfg["sim"]["dt"], cfg["sim"]["substeps"], precision="f32", threads=threads, ground_mu=e["terrain"]["dynamicFriction"],
                    hfield=hs.astype(np.float64) * ter.vertical_scale, hf_scale=ter.horizontal_scale, hf_origin=(-ter.border_size, -ter.border_size))
    rng = np.random.default_rng(42)
    names = list(m.dof_names)
    q0 = np.array([e["defaultJointAngles"][nme] for nme in names], f32)
    dec = int(e["control"]["decimation"]); dt = dec * cfg["sim"]["dt"]
    Kp, Kd, sc = f32(e["control"]["stiffness"]), f32(e["control"]["damping"]), f32(e["control"]["actionScale"])
    keys = [("termination", "terminalReward"), ("lin_vel_xy", "linearVelocityXYRewardScale"), ("lin_vel_z", "linearVelocityZRewardScale"),
            ("ang_vel_z", "angularVelocityZRewardScale"), ("ang_vel_xy", "angularVelocityXYRewardScale"), ("orient", "orientationRewardScale"),
            ("torque", "torqueRewardScale"), ("joint_acc", "jointAccRewardScale"), ("base_height", "baseHeightRewardScale"),
            ("air_time", "feetAirTimeRewardScale"), ("collision", "kneeCollisionRewardScale"), ("stumble", "feetStumbleRewardScale"),
            ("action_rate", "actionRateRewardScale"), ("hip", "hipRewardScale")]
    rs = {k: learn[y] * dt for k, y in keys}
    max_len = int(learn["episodeLength_s"] / dt + 0.5)
    org = np.asarray(ter.env_origins, f32)[rng.integers(0, e["terrain"]["maxInitMapLevel"] + 1, n_envs), rng.integers(0, e["terrain"]["numTerrains"], n_envs)]
    b = e["baseInitState"]
    base = np.array(b["pos"] + b["rot"] + b["vLinear"] + b["vAngular"], f32)
    root = np.tile(base, (n_envs, 1)); root[:, :3] += org
    dof = np.zeros((n_envs, 12, 2), f32); dof[..., 0] = q0
    st = dict(progress=np.zeros(n_envs, np.int64), last_a=np.zeros((n_envs, 12), f32), last_v=np.zeros((n_envs, 12), f32),
              fat=np.zeros((n_envs, 4), f32), cmd=np.zeros((n_envs, 4), f32))
    st["cmd"][:, 0] = rng.uniform(-1, 1, n_envs); st["cmd"][:, 3] = rng.uniform(-3.14, 3.14, n_envs)
    body_names = list(m.body_names)
    feet = [i for i, s in enumerate(body_names) if e["urdfAsset"]["footName"] in s]
    knees = [i for i, s in enumerate(body_names) if e["urdfAsset"]["kneeName"] in s]

    def one():
        a = np.clip(rng.uniform(-1, 1, size=(n_envs, 12)).astype(f32), -100, 100)
        tau = None
        for _ in range(dec):
            tau = np.clip(Kp * (sc * a + q0[None] - dof[..., 0]) - Kd * dof[..., 1], -80.0, 80.0).astype(f32)
            out = sim.simulate(root, dof, tau)
        out = sim.simulate(root, dof, tau)                       # controlFrequencyInv = 1 (vec_task.py:379-382)
        st["progress"] += 1
        cf = out["contact_force"].astype(f32)
        blv, bav, pg, cmd = T.anymal_prepare(root, st["cmd"])
        reset = T.anymal_check_termination(cf, st["progress"], max_len, base_index=body_names.index("base"), knee_indices=knees,
                                           allow_knee_contacts=learn["allowKneeContacts"])
        timeout = st["progress"] >= max_len - 1
        rew, st["fat"], _ = T.anymal_reward(blv, bav, pg, cmd, root, tau, st["last_v"], dof[..., 1], dof[..., 0], q0, cf, st["last_a"], a,
                                            st["fat"], reset, timeout, rs, dt, knee_indices=knees, feet_indices=feet)
        ids = np.nonzero(reset)[0]
        if len(ids):
            dof[ids, :, 0] = q0 * rng.uniform(0.5, 1.5, size=(len(ids), 12)).astype(f32)
            dof[ids, :, 1] = rng.uniform(-0.1, 0.1, size=(len(ids), 12)).astype(f32)
            root[ids] = base; root[ids, :3] += org[ids]
            st["progress"][ids] = 0; st["fat"][ids] = 0
        hts = T.anymal_get_heights(root, hs, ter.border_size, ter.horizontal_scale, ter.vertical_scale)
        T.anymal_observations(blv, bav, pg, cmd, dof[..., 0], dof[..., 1], root, hts, a)
        st["cmd"] = cmd; st["last_a"] = a; st["last_v"] = dof[..., 1].copy()
    return one


def _hand_cpu(n_envs, threads):
    """ShadowHand control step on host cores: oracle physics of hand + cube, numpy restatement of the task."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from tests.hand_common import hand_setup, DT, SUBSTEPS, G
    from oracle.oracle import OracleSim
    from oracle import tasks_np as T
    f32 = np.float32
    m, obj, tendons = hand_setup()
    sim = OracleSim(m, DT, SUBSTEPS, G, precision="f32", obj=obj, tendons=tendons, tendon_k=30.0, tendon_d=0.1, threads=threads)
    D = m.ndof
    names = list(m.dof_names)
    rng = np.random.default_rng(42)
    root = np.zeros((n_envs, 3, 13), f32); root[:, :, 6] = 1
    root[:, 0, 0:3] = [0, 0, 0.5]; root[:, 0, 3:7] = m.default_root_quat
    obj_init = np.zeros((n_envs, 13), f32); obj_init[:, 0:3] = [0, -0.39, 0.6]; obj_init[:, 6] = 1
    goal_init = obj_init.copy(); goal_init[:, 2] -= 0.04
    st = dict(root=root, dof_pos=np.zeros((n_envs, D), f32), dof_vel=np.zeros((n_envs, D), f32), cur_targets=np.zeros((n_envs, D), f32),
              prev_targets=np.zeros((n_envs, D), f32), goal_states=goal_init.copy(), reset=np.ones(n_envs, np.int64),
              reset_goal=np.ones(n_envs, np.int64), progress=np.zeros(n_envs, np.int64), successes=np.zeros(n_envs, f32),
              reset_count=np.zeros(n_envs, np.int32), goal_reset_count=np.zeros(n_envs, np.int32))
    P = dict(seed=42, goal_init=goal_init, object_init=obj_init, goal_displacement=f32([-0.2, -0.06, 0.12]), reset_position_noise=0.01,
             reset_dof_pos_noise=0.2, reset_dof_vel_noise=0.0, lower=m.lower[1:].astype(f32), upper=m.upper[1:].astype(f32),
             default_pos=np.zeros(D, f32), default_vel=np.zeros(D, f32), clip_actions=1.0,
             actuated=np.array([names.index(j) for j in m.actuator_joint]), use_relative_control=False, dof_speed_scale=20.0, dt=DT,
             act_moving_average=1.0, obs_type="full_state", vel_obs_scale=0.2, force_torque_obs_scale=10.0, dist_reward_scale=-10.0,
             rot_reward_scale=1.0, rot_eps=0.1, action_penalty_scale=-0.0002, success_tolerance=0.1, reach_goal_bonus=250.0,
             fall_dist=0.24, fall_penalty=0.0, max_consecutive_successes=0, max_episode_length=600.0, av_factor=0.1)
    box = dict(cons=f32(0))
    ft_idx = m.sensor_body

    def one():
        a = T.hand_pre_physics(st, rng.uniform(-1, 1, size=(n_envs, 20)).astype(f32), P)
        hand = np.ascontiguousarray(st["root"][:, 0]); o = np.ascontiguousarray(st["root"][:, 1])
        dof = np.ascontiguousarray(np.stack([st["dof_pos"], st["dof_vel"]], -1))
        out = sim.simulate(hand, dof, target=st["cur_targets"], obj=o)
        st["root"][:, 1] = o; st["dof_pos"][:] = dof[..., 0]; st["dof_vel"][:] = dof[..., 1]
        st["progress"] += 1
        ft = out["body_state"][:, ft_idx]
        T.hand_observations(st, a, ft, out["sensor"], out["dof_force"], P)
        _, box["cons"] = T.hand_reward(st, a, box["cons"], P)
    return one


def cpu_pipeline(task, n_envs, steps, threads, warmup=1):
    """K control steps of `task` over n_envs envs on host cores.  -> (env-steps/s, seconds)."""
    if task in ("Ant", "Humanoid"):
        one = _loco_cpu(task, n_envs, threads)
    elif task == "Cartpole":
        one = _cartpole_cpu(n_envs, threads)
    elif task == "AnymalTerrain":
        one = _anymal_cpu(n_envs, threads)
    else:
        one = _hand_cpu(n_envs, threads)
    for _ in range(max(1, warmup)):
        one()
    t0 = time.perf_counter()
    for _ in range(steps):
        one()
    dt = time.perf_counter() - t0
    return n_envs * steps / dt, dt


CPU_WHAT = "oracle/aba_oracle.c f32 physics (pthreads over envs) + oracle/tasks_np.py obs/reward (numpy); the reference's own sim_device=cpu path needs the closed Isaac Gym binary"


def run_reference_arm(args):
    """`--impl reference`: the reference's CPU pipeline cannot run here (closed Isaac Gym binary, SURVEY.md 8c), so this
    arm times the CPU PORT of the path (oracle/) on all host cores, on the SAME config as the GPU arm (same env count)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    task, n_full, _ = WORKLOADS[args.workload]
    n = args.num_envs or n_full
    cores = os.cpu_count() or 1
    k = args.steps                                          # each step is the whole workload
    v, secs = cpu_pipeline(task, n, k, cores, warmup=max(1, min(args.warmup, 3)))
    line = {"metric": METRIC, "impl": "reference", "value": v, "unit": "env-steps/s", "n_gpus": args.gpus,
            "steps": k, "warmup": args.warmup, "ms_per_step": 1e3 * secs / k,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"{task} num_envs={n} random actions U(-1,1)", "sample_envs": n, "same_config": True,
                       "steps_requested": args.steps},
            "cpu_baseline": {"value": v, "unit": "env-steps/s", "cores": cores, "kind": "port",
                             "sample": f"{n} envs x {k} control steps, {secs:.1f} s ({CPU_WHAT})"},
            "e2e": {"value": v, "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------ GPU arm
DUMP_LIMIT_BYTES = 64 * 1024 * 1024


def step_outputs(result):
    """What VecTask.step() hands its caller (obs dict, reward, reset, the tensors in extras) as float32 / float64 host arrays."""
    import torch
    obs_dict, rew, reset, extras = result
    named = dict(obs_dict)
    named.update(rew=rew, reset=reset)
    named.update({k: v for k, v in extras.items() if torch.is_tensor(v)})
    return {k: (v.double() if v.dtype == torch.float64 else v.float()).cpu().numpy() for k, v in named.items()}


def dump_outputs(outputs, out_dir):
    """Writes out_dir/<name>.npy.  Above DUMP_LIMIT_BYTES in all, every per-env array keeps the same fixed, seeded sample of
    envs, whose indices go to sample_envs.npy."""
    n = outputs["rew"].shape[0]
    total = sum(a.nbytes for a in outputs.values())
    if total > DUMP_LIMIT_BYTES:
        per_env = sum(a.nbytes for a in outputs.values() if a.ndim and a.shape[0] == n) / n
        keep = int((DUMP_LIMIT_BYTES - (total - per_env * n) - 8 * n) // per_env)
        rows = np.sort(np.random.default_rng(0).choice(n, size=keep, replace=False))
        outputs = {k: (a[rows] if a.ndim and a.shape[0] == n else a) for k, a in outputs.items()}
        outputs["sample_envs"] = rows.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for name, a in outputs.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def run_gpu_arm(args):
    import torch
    import torch.distributed as dist
    from isaacgymenvs_b200 import distributed as D
    rank, local, world = D.rank_info()
    torch.cuda.set_device(local)
    D.init("nccl")
    device = f"cuda:{local}"
    task, n, bytes_per = WORKLOADS[args.workload]
    if args.num_envs:
        n = args.num_envs
    if args.scaling == "strong":
        assert n % world == 0
        n = n // world                                  # the same total env count split over the ranks
    # Timing hygiene: inputs larger than L2.  One env set's live tensors (n * bytes_per, ~11 MB for Ant) would stay
    # L2-resident between steps, so the bench steps R independent env sets round-robin with R * n * bytes_per >= 1.5 x L2:
    # by the time a set is stepped again, everything it reads has been evicted and comes from HBM, while the kernel's
    # code stays warm, as in a real rollout loop.
    L2_BYTES = 126 * 1024 * 1024
    R = args.sets if args.sets > 0 else max(2, -(-int(1.5 * L2_BYTES) // (n * bytes_per)))
    R = min(R, 192)
    envs = [make_env(task, n, device, rank) for _ in range(R)]
    env = envs[0]
    A = env.num_actions
    gen = torch.Generator(device=device).manual_seed(42 + rank)
    ring = [2 * torch.rand((n, A), device=device, generator=gen) - 1 for _ in range(16)]
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=device)   # > 126 MB L2

    def barrier():
        D.barrier()
        torch.cuda.synchronize()

    for k in range(args.warmup):
        for ev_ in envs:
            ev_.step(ring[k % 16])
    barrier()
    sampler = ClockSampler(local); sampler.start()
    l0 = sum(e_.sim.launch_count() for e_ in envs)
    barrier()
    # ---- headline: K x VecTask.step() round-robin over the R sets, one CUDA-event pair around all of them
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    w0 = time.perf_counter()
    t0.record()
    for k in range(args.steps):
        last = envs[k % R].step(ring[k % 16])
    t1.record()
    host_issue_s = time.perf_counter() - w0                 # host time to ISSUE the K steps (no sync inside)
    barrier()
    launches = sum(e_.sim.launch_count() for e_ in envs) - l0
    total_ms = t0.elapsed_time(t1)
    # the env buffers are stepped again below: copy the last timed step's results out now
    outputs = step_outputs(last) if args.dump_outputs else None
    # ---- device only: the same K steps as bare C-ABI launches (b2g_task_step), same rotation: the kernel time
    d0, d1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    d0.record()
    for k in range(args.steps):
        envs[k % R].sim.task_step(ring[k % 16])
    d1.record()
    barrier()
    dev_ms = d0.elapsed_time(d1)
    # ---- same K steps on ONE set with an explicit L2 flush between steps (also evicts the kernel's code): per-step events
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    sink = torch.zeros(1, device=device)
    for k in range(args.steps):
        flush.zero_()                      # write 256 MB (> 126 MB L2): evicts the previous step's tensors ...
        sink += flush.sum()                # ... then read it back: the dirty lines are written out, L2 is left clean and cold
        ev[k][0].record()
        env.sim.task_step(ring[k % 16])
        ev[k][1].record()
    barrier()
    flushed_ms = float(sum(a.elapsed_time(b) for a, b in ev))
    # ---- back-to-back (no flush) over the same K steps: what a rollout loop with a tiny policy sees
    s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    s0.record()
    for k in range(args.steps):
        env.sim.task_step(ring[k % 16])
    s1.record()
    barrier()
    b2b_ms = s0.elapsed_time(s1)
    # ---- open-loop rollout: VecTask.rollout((KR, n, A) actions) -- KR steps per launch where the task has the fused form (Ant)
    KR = 16
    roll_ms, roll_calls = None, 0
    if task == "Ant" and not args.no_rollout:
        acts = torch.stack(ring[:KR]).contiguous()
        for ev_ in envs[:min(R, 4)]:
            ev_.rollout(acts)
        roll_calls = max(1, -(-args.steps // KR))
        barrier()
        r0, r1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        r0.record()
        for j in range(roll_calls):
            envs[j % R].rollout(acts)
        r1.record()
        barrier()
        roll_ms = r0.elapsed_time(r1)
    # ---- end to end through the public API with HOST buffers (pinned): H2D actions, step, D2H results
    O = env.num_obs
    h_a = [r.cpu().pin_memory() for r in ring]
    h_obs = torch.zeros(n, O).pin_memory(); h_rew = torch.zeros(n).pin_memory()
    h_reset = torch.zeros(n, dtype=torch.long).pin_memory(); h_to = torch.zeros(n, dtype=torch.uint8).pin_memory()
    for k in range(max(3, args.warmup)):
        env.step_host(h_a[k % 16], h_obs, h_rew, h_reset, h_to)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for k in range(args.steps):
        env.step_host(h_a[k % 16], h_obs, h_rew, h_reset, h_to)
    e1.record()
    barrier()
    e2e_ms = e0.elapsed_time(e1)
    clocks = sampler.stop()
    # ---- logging collective: per-env returns gathered once per rollout (north_star), off the step path
    all_returns = D.gather_returns(env.rew_buf)           # (world*n,) in global env order
    assert all_returns.numel() == world * n
    # ---- max over ranks
    total_ms, dev_ms, b2b_ms, e2e_ms, flushed_ms, roll_max = D.max_over_ranks([total_ms, dev_ms, b2b_ms, e2e_ms, flushed_ms, roll_ms or 0.0], device=device)
    roll_ms = roll_max if roll_ms is not None else None
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    value = world * n * args.steps / (total_ms * 1e-3)
    peak, peak_kind = measured_peak()
    kernel_ms = dev_ms / args.steps
    achieved = n * bytes_per / (kernel_ms * 1e-3) / 1e9
    traffic, flop = None, None
    try:
        with open(os.path.join(ROOT, "profiles", "roofline_traffic.json")) as f:
            prof = json.load(f)
        traffic = prof.get(args.workload)
        flop = prof.get(args.workload + "_fp32_flop_per_launch")
    except Exception:
        pass
    if flop is not None and n != WORKLOADS[args.workload][1]:
        flop = flop * n / WORKLOADS[args.workload][1]
    quad = env.sim.quad_ns()
    line = {
        "metric": METRIC, "value": value, "unit": "env-steps/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": total_ms / args.steps, "higher_is_better": True, "scaling": args.scaling,
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"{task} num_envs={n} per GPU, random actions U(-1,1), sim dt {env.cfg['sim']['dt']} x {env.cfg['sim']['substeps']} substeps",
                   "num_envs_total": world * n, "env_sets": R,
                   "timing": f"value = K x VecTask.step(actions) (device tensors) inside one CUDA-event pair on the launching stream; inputs larger than L2: {R} independent env sets of {n} envs stepped round-robin ({R * n * bytes_per / 1e6:.0f} MB of live tensors > 126 MB L2), so every step reads its state from HBM",
                   "collective": "none on the step path; one NCCL all_gather of per-env returns per rollout (logging)",
                   "substep_formulation": f"quad (4 chains x {quad})" if quad else "generic slot program",
                   "parity": PARITY_NOTE},
        "api": {"call": "VecTask.step(actions)", "ms_per_step": total_ms / args.steps, "host_issue_ms_per_step": 1e3 * host_issue_s / args.steps,
                "vs_device_only": (total_ms / dev_ms)},
        "device_only": {"value": world * n * args.steps / (dev_ms * 1e-3), "unit": "env-steps/s", "ms_per_step": kernel_ms,
                        "note": "the same K steps as bare b2g_task_step launches (no Python task layer): the kernel's own duration"},
        "l2_flushed": {"value": world * n * args.steps / (flushed_ms * 1e-3), "unit": "env-steps/s", "ms_per_step": flushed_ms / args.steps,
                       "note": "one env set, per-step events, L2 flushed between steps by writing and reading back a 256 MB buffer (evicts the kernel's code too)"},
        "back_to_back": {"value": world * n * args.steps / (b2b_ms * 1e-3), "unit": "env-steps/s", "ms_per_step": b2b_ms / args.steps,
                         "note": "same K steps on one env set (state stays L2-resident)"},
        "e2e": {"value": world * n * args.steps / (e2e_ms * 1e-3), "unit": "env-steps/s",
                "h2d_bytes_per_step": n * A * 4, "d2h_bytes_per_step": n * (O * 4 + 4 + 8 + 1), "ms_per_step": e2e_ms / args.steps},
        "gpu_launches": int(launches),
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": traffic, "peak_kind": peak_kind, "kernel_ms": kernel_ms,
                     "algorithmic_bytes_per_env_step": bytes_per},
        "clocks": clocks,
    }
    if roll_ms is not None:
        line["rollout"] = {"call": f"VecTask.rollout(actions[{KR}, n, A])", "value": world * n * roll_calls * KR / (roll_ms * 1e-3), "unit": "env-steps/s",
                           "ms_per_step": roll_ms / (roll_calls * KR), "steps_per_launch": KR,
                           "note": "open-loop (random-action) rollout, the README benchmark's shape: all KR actions given up front, state stays on chip "
                                   "between the steps, every step's obs/reward/reset/time_out written to (KR, n, .) outputs; NOT the headline: a policy in "
                                   "the loop needs step()"}
    if flop is not None:    # SURVEY 8d cross-check: the kernel is FP32-issue-bound, not HBM-bound
        tf = flop / (kernel_ms * 1e-3) / 1e12
        line["roofline"]["fp32"] = {"flop_per_launch": flop, "achieved": tf, "peak": 74.4, "unit": "TFLOP/s", "frac": tf / 74.4,
                                    "note": "FFMA x2 + FADD + FMUL thread-instructions from the ncu capture in profiles/; peak = 148 SM x 128 lanes x 2 x 1.965 GHz"}
    if world == 1 and not args.no_cpu_baseline:
        cores = os.cpu_count() or 1
        est = {"Ant": 0.8e6, "Humanoid": 0.25e6, "Cartpole": 4e6, "AnymalTerrain": 0.15e6, "ShadowHand": 0.3e6}[task] * cores / 128.0
        ks = max(3, min(200, int(15.0 * est / n)))          # the workload's own env count for ~15 s of CPU work
        v, secs = cpu_pipeline(task, n, ks, cores)
        line["cpu_baseline"] = {"value": v, "unit": "env-steps/s", "cores": cores, "kind": "port",
                                "sample": f"{n} envs x {ks} control steps, {secs:.1f} s ({CPU_WHAT})"}
    if outputs is not None:
        dump_outputs(outputs, args.dump_outputs)
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2000)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="ant", choices=sorted(WORKLOADS))
    ap.add_argument("--num-envs", type=int, default=0)
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="weak: the workload's env count on EVERY GPU; strong: the same total split over the GPUs")
    ap.add_argument("--sets", type=int, default=0, help="independent env sets stepped round-robin (0 = enough to exceed 1.5 x L2)")
    ap.add_argument("--no-rollout", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed VecTask.step() returned as DIR/<name>.npy (same arguments, same inputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the GPU path; the reference arm has none to give")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_gpu_arm(args)


if __name__ == "__main__":
    main()
