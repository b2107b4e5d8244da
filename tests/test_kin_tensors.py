"""Jacobian and mass-matrix tensors (gym.acquire_jacobian_tensor / acquire_mass_matrix_tensor, reference call sites
tasks/franka_cube_stack.py:388-392, consumed by the operational-space controller :600-627).

CPU half: pins the oracle's restatement (oracle/aba_oracle.c "kinematic / inertial tensors") against things that share
no code with it -- the rigid-body-state twists of the oracle's forward kinematics, central differences of body positions,
and the independent Newton-Euler inverse dynamics of tests/rnea_np.py (column j of M = the forces REQUIRED by a unit
acceleration of coordinate j at rest, without gravity).  GPU half: the CUDA kernel (csrc/b2g_kin.cuh) against the oracle.
"""
import numpy as np
import pytest

from isaacgymenvs_b200.assets import load_compiled
from oracle.oracle import OracleSim
from tests import rnea_np
from tests.test_oracle_physics import random_state

MODELS = ["cartpole", "ant", "humanoid", "anymal", "shadow_hand", "franka"]


def _states(m, n, seed):
    rng = np.random.default_rng(seed)
    rs, ds = zip(*[random_state(m, rng) for _ in range(n)])
    return np.stack(rs), np.stack(ds)


def _gen_vel(m, root, dof):
    """generalised velocity in the tensors' column order: (world linear, world angular of the root origin), joints"""
    qd = dof[:, :, 1]
    return qd if m.root_fixed else np.concatenate([root[:, 7:13], qd], 1)


@pytest.mark.parametrize("name", MODELS)
def test_oracle_jacobian_reproduces_rigid_body_twists(name):
    m = load_compiled(name)
    orc = OracleSim(m, 0.0166, 2)
    root, dof = _states(m, 8, 1)
    J = orc.jacobian(root, dof)
    rows, _, nc = orc.jacobian_shape()
    assert J.shape == (8, rows, 6, nc) and rows == (m.nb - 1 if m.root_fixed else m.nb) and nc == m.ndof + (0 if m.root_fixed else 6)
    tw = np.einsum("nbrc,nc->nbr", J, _gen_vel(m, root, dof))
    bs = orc.body_states(root, dof)[:, (1 if m.root_fixed else 0):]
    assert np.abs(tw[..., :3] - bs[..., 7:10]).max() < 1e-10 and np.abs(tw[..., 3:] - bs[..., 10:13]).max() < 1e-10


@pytest.mark.parametrize("name", MODELS)
def test_oracle_jacobian_is_the_derivative_of_body_positions(name):
    m = load_compiled(name)
    orc = OracleSim(m, 0.0166, 2)
    root, dof = _states(m, 3, 2)
    J = orc.jacobian(root, dof)
    off, nb0, eps = (0 if m.root_fixed else 6), (1 if m.root_fixed else 0), 1e-6
    for j in range(m.ndof):
        dp, dm = dof.copy(), dof.copy()
        dp[:, j, 0] += eps; dm[:, j, 0] -= eps
        fd = (orc.body_states(root, dp)[:, nb0:, :3] - orc.body_states(root, dm)[:, nb0:, :3]) / (2 * eps)
        assert np.abs(fd - J[:, :, :3, off + j]).max() < 1e-8, (name, j)
    if not m.root_fixed:          # base translation columns; the base rotation columns are covered by the twist identity
        for k in range(3):
            rp, rm = root.copy(), root.copy()
            rp[:, k] += eps; rm[:, k] -= eps
            fd = (orc.body_states(rp, dof)[:, :, :3] - orc.body_states(rm, dof)[:, :, :3]) / (2 * eps)
            assert np.abs(fd - J[:, :, :3, k]).max() < 1e-8


@pytest.mark.parametrize("name", MODELS)
def test_oracle_mass_matrix_columns_are_inverse_dynamics_of_unit_accelerations(name):
    m = load_compiled(name)
    orc = OracleSim(m, 0.0166, 2)
    root, dof = _states(m, 2, 3)
    dof[:, :, 1] = 0; root[:, 7:] = 0
    M = orc.mass_matrix(root, dof)
    nb = 0 if m.root_fixed else 6
    nc = m.ndof + nb
    assert M.shape == (2, nc, nc)
    z3 = np.zeros(3)
    for e in range(2):
        q = dof[e, :, 0]
        col = np.zeros((nc, nc))
        for j in range(nc):
            qdd = np.zeros(m.ndof); acc = [z3.copy(), z3.copy()]
            if j < nb:
                acc[j // 3][j % 3] = 1.0
            else:
                qdd[j - nb] = 1.0
            tau, (f0, n0) = rnea_np.inverse_dynamics(m, root[e], q, np.zeros(m.ndof), qdd, tuple(acc), (0.0, 0.0, 0.0))
            col[nb:, j] = tau
            if nb:
                col[:3, j], col[3:6, j] = f0, n0
        col[np.arange(nb, nc), np.arange(nb, nc)] += m.armature[1:]
        scale = np.abs(col).max()
        assert np.abs(M[e] - col).max() < 1e-10 * max(1.0, scale), name
        assert np.abs(M[e] - M[e].T).max() < 1e-12 * max(1.0, scale)
        assert np.linalg.eigvalsh(M[e]).min() > 0


def test_oracle_kinetic_energy_is_the_quadratic_form_of_the_mass_matrix():
    m = load_compiled("humanoid")
    orc = OracleSim(m, 0.0166, 2)
    root, dof = _states(m, 4, 4)
    M = orc.mass_matrix(root, dof)
    u = _gen_vel(m, root, dof)
    ke = 0.5 * np.einsum("ni,nij,nj->n", u, M - np.diag(np.r_[np.zeros(6), m.armature[1:]])[None], u)
    from isaacgymenvs_b200.importer import rot
    for e in range(4):
        R, x, v, w, *_ = rnea_np.kinematics(m, root[e], dof[e, :, 0], dof[e, :, 1], np.zeros(m.ndof), (np.zeros(3), np.zeros(3)))
        t = 0.0
        for i in range(m.nl):
            c = R[i] @ m.com[i]; vc = v[i] + np.cross(w[i], c)
            Iw = R[i] @ rot.sym6_to_mat(m.inertia[i]) @ R[i].T
            t += 0.5 * m.mass[i] * vc @ vc + 0.5 * w[i] @ Iw @ w[i]
        assert abs(t - ke[e]) < 1e-9 * max(1.0, t)


# ---------------------------------------------------------------------------------------------------------------
# the device arithmetic on the CPU (tests/kin_host.cu compiles csrc/b2g_kin.cuh for the host) against the oracle
import ctypes as C
import os
import subprocess

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
KSRC, KLIB = os.path.join(HERE, "kin_host.cu"), os.path.join(HERE, "libkinhost.so")
KDEPS = [KSRC] + [os.path.join(ROOT, "isaacgymenvs_b200", "csrc", f) for f in ("b2g_kin.cuh", "b2g_kin_host.h", "b2g_device.cuh")]

# fp32 kernel arithmetic vs the fp64 oracle: J entries are O(1) lengths / unit vectors, M is compared relative to its largest entry
J_TOL, M_RTOL = 2e-5, 2e-5


def _klib():
    if not os.path.exists(KLIB) or any(os.path.getmtime(d) > os.path.getmtime(KLIB) for d in KDEPS):
        nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
        subprocess.check_call([nvcc, "-O2", "-std=c++17", "--expt-relaxed-constexpr", "-Wno-deprecated-gpu-targets", "-shared",
                               "-Xcompiler", "-fPIC", "-o", KLIB, KSRC])
    return C.CDLL(KLIB)


def _host_tensors(m, root, dof):
    from isaacgymenvs_b200 import engine
    lib = _klib()
    cm, keep = engine.pack_model(m)
    rows, nc = C.c_int(), C.c_int()
    assert lib.kin_host_shape(C.byref(cm), C.byref(rows), C.byref(nc)) == 0
    N = root.shape[0]
    r32, d32 = np.ascontiguousarray(root, np.float32), np.ascontiguousarray(dof, np.float32)
    J = np.full((N, rows.value, 6, nc.value), np.nan, np.float32); M = np.full((N, nc.value, nc.value), np.nan, np.float32)
    p = lambda a: C.c_void_p(a.ctypes.data)
    assert lib.kin_host_tensors(C.byref(cm), C.c_int(1), C.c_int(N), p(r32), p(d32), p(J), p(M)) == 0
    return J, M


@pytest.mark.parametrize("name", MODELS)
def test_device_arithmetic_on_the_host_matches_oracle(name):
    m = load_compiled(name)
    orc = OracleSim(m, 0.0166, 2)
    root, dof = _states(m, 64, 5)
    J, M = _host_tensors(m, root, dof)
    Jo, Mo = orc.jacobian(root, dof), orc.mass_matrix(root, dof)
    assert J.shape == Jo.shape and M.shape == Mo.shape
    assert np.abs(J - Jo).max() < J_TOL, np.abs(J - Jo).max()
    assert np.abs(M - Mo).max() < M_RTOL * np.abs(Mo).max(), (np.abs(M - Mo).max(), np.abs(Mo).max())


# ---------------------------------------------------------------------------------------------------------------
# GPU: the CUDA kernel through the C ABI (b2g_refresh_kinematic_tensors) against the oracle
def _gpu_sim(name, n):
    import torch
    from isaacgymenvs_b200 import engine
    m = load_compiled(name)
    if name == "shadow_hand":            # three actors per env: the kernel must step over the object's and the goal's root rows
        from tests.hand_common import hand_setup, DT, SUBSTEPS, G as HG
        m, obj, tendons = hand_setup()
        ext = engine.pack_model_ext(m, obj=obj, actors_per_env=3, tendons=tendons, tendon_k=30.0, tendon_d=0.1)
        return m, engine.Sim(m, n, DT, SUBSTEPS, HG, ground_mu=1.0, ext=ext), 3
    return m, engine.Sim(m, n, 0.0166, 2, (0.0, 0.0, -9.81)), 1


@pytest.mark.gpu
@pytest.mark.parametrize("name,n", [("cartpole", 1001), ("ant", 16384), ("humanoid", 8192), ("anymal", 4099), ("shadow_hand", 4096)])
def test_gpu_kinematic_tensors_match_oracle(name, n):
    import torch
    from isaacgymenvs_b200 import engine
    m, sim, stride = _gpu_sim(name, n)
    ncheck = 256                                       # the oracle is evaluated on a spread sample, the kernel on all n envs
    root, dof = _states(m, ncheck, 6)
    idx = np.linspace(0, n - 1, ncheck).astype(np.int64)
    rs = np.zeros((n, stride, 13), np.float32); rs[..., 6] = 1.0
    rs[idx, 0] = root
    ds = np.zeros((n, m.ndof, 2), np.float32); ds[idx] = dof
    sim.root_state.copy_(torch.tensor(rs.reshape(-1, 13)))
    sim.dof_state.copy_(torch.tensor(ds.reshape(-1, 2)))
    J, M = sim.refresh_kinematic_tensors()
    torch.cuda.synchronize()
    orc = OracleSim(m, 0.0166, 2)
    rows, _, nc = orc.jacobian_shape()
    assert sim.kin_shape() == (rows, nc) and tuple(J.shape) == (n, rows, 6, nc) and tuple(M.shape) == (n, nc, nc)
    # the oracle sees the float32 state the kernel saw
    Jo = orc.jacobian(rs[idx, 0].astype(np.float64), ds[idx].astype(np.float64))
    Mo = orc.mass_matrix(rs[idx, 0].astype(np.float64), ds[idx].astype(np.float64))
    Jg, Mg = J.cpu().numpy(), M.cpu().numpy()
    assert np.isfinite(Jg).all() and np.isfinite(Mg).all()
    assert np.abs(Jg[idx] - Jo).max() < J_TOL, np.abs(Jg[idx] - Jo).max()
    assert np.abs(Mg[idx] - Mo).max() < M_RTOL * np.abs(Mo).max(), (np.abs(Mg[idx] - Mo).max(), np.abs(Mo).max())
    # ... and equals the host twin of the same arithmetic up to FMA contraction and the library sincos (deep chains accumulate it)
    Jh, Mh = _host_tensors(m, rs[idx, 0], ds[idx])
    assert np.abs(Jg[idx] - Jh).max() < 5e-6 and np.abs(Mg[idx] - Mh).max() < 1e-5 * np.abs(Mo).max()
    # size-independent properties on ALL envs: symmetric positive-definite M; the twist J u of every body equals the
    # rigid-body-state tensor's velocities (forward-kinematics kernel, independent code)
    assert float((M - M.transpose(1, 2)).abs().max()) <= 1e-6 * float(M.abs().max())
    assert float(torch.linalg.eigvalsh(M.double()).min()) > 0
    # one kernel refreshes either tensor alone
    J.zero_(); sim.refresh_kinematic_tensors(jacobian=True, mass_matrix=False); torch.cuda.synchronize()
    assert np.array_equal(J.cpu().numpy(), Jg)
    u = sim.dof_state.view(n, m.ndof, 2)[:, :, 1]
    if not m.root_fixed:
        u = torch.cat([sim.root_state.view(n, stride, 13)[:, 0, 7:13], u], 1)
    tw = torch.einsum("nbrc,nc->nbr", J, u)
    bs = sim.refresh_rigid_body_state().view(n, -1, 13)[:, (1 if m.root_fixed else 0):m.nb]
    torch.cuda.synchronize()
    scale = max(1.0, float(bs[..., 7:13].abs().max()))
    assert float((tw[..., :3] - bs[..., 7:10]).abs().max()) < 2e-5 * scale
    assert float((tw[..., 3:] - bs[..., 10:13]).abs().max()) < 2e-5 * scale


@pytest.mark.gpu
def test_compat_gym_jacobian_and_mass_matrix_calls():
    """the reference's call sequence (franka_cube_stack.py:388-392, 439-440) through the compatibility shim, on the Ant
    (floating base: six base columns first); the operational-space inertia of a foot, (J M^-1 J^T)^-1 as the controller
    forms it (:603-605), is finite and symmetric positive definite"""
    import torch
    from isaacgymenvs_b200 import compat
    compat.install()
    from isaacgym import gymapi, gymtorch
    gym = gymapi.acquire_gym()
    sp = gymapi.SimParams(); sp.dt, sp.substeps, sp.up_axis, sp.gravity, sp.use_gpu_pipeline = 0.0166, 2, gymapi.UP_AXIS_Z, gymapi.Vec3(0, 0, -9.81), True
    sim = gym.create_sim(0, -1, gymapi.SIM_PHYSX, sp)
    gym.add_ground(sim, gymapi.PlaneParams())
    ao = gymapi.AssetOptions(); ao.angular_damping = 0.0
    asset = gym.load_asset(sim, "/no/such/checkout/assets/mjcf", "nv_ant.xml", ao)
    n = 64
    pose = gymapi.Transform(); pose.p = gymapi.Vec3(0, 0, 0.44)
    for i in range(n):
        e = gym.create_env(sim, gymapi.Vec3(-5, -5, 0), gymapi.Vec3(5, 5, 5), 8)
        gym.create_actor(e, asset, pose, "ant", i, 1, 0)
    gym.prepare_sim(sim)
    jac = gymtorch.wrap_tensor(gym.acquire_jacobian_tensor(sim, "ant"))
    mm = gymtorch.wrap_tensor(gym.acquire_mass_matrix_tensor(sim, "ant"))
    nd, nb = gym.get_asset_dof_count(asset), gym.get_asset_rigid_body_count(asset)
    assert tuple(jac.shape) == (n, nb, 6, nd + 6) and tuple(mm.shape) == (n, nd + 6, nd + 6)
    dof = gymtorch.wrap_tensor(gym.acquire_dof_state_tensor(sim)).view(n, nd, 2)
    dof[:, :, 0] = 0.3 * (torch.rand(n, nd, device=dof.device) - 0.5)
    assert gym.refresh_jacobian_tensors(sim) and gym.refresh_mass_matrix_tensors(sim)
    foot = [i for i, s in enumerate(gym.get_asset_rigid_body_names(asset)) if "foot" in s][0]
    j_eef = jac[:, foot, :3]
    m_eef_inv = j_eef @ torch.inverse(mm) @ j_eef.transpose(1, 2)
    assert torch.isfinite(m_eef_inv).all() and float(torch.linalg.eigvalsh(m_eef_inv.double()).min()) > 0
    # total mass on the base block's linear diagonal
    mass = float(load_compiled("ant").mass.sum())
    assert abs(float(mm[0, 0, 0]) - mass) < 1e-5 * mass and abs(float(mm[0, 2, 2]) - mass) < 1e-5 * mass


@pytest.mark.parametrize("name", ["cartpole", "ant", "humanoid", "anymal"])
def test_mass_matrix_is_the_inertia_the_aba_step_inverts(name):
    """The oracle's mass matrix (CRBA) against the oracle's articulated-body algorithm (an O(n) recursion that never forms M):
    from rest, without gravity and off the ground, one sub-step's accelerations a satisfy
        (M + diag(h b + h^2 k)) a = (0 ; clip(tau) - k q)
    -- the implicit joint damping / stiffness terms of the scheme (DESIGN.md section 3) join the diagonal, nothing else."""
    m = load_compiled(name)
    dt, sub = 0.0166, 2
    h = dt / sub
    orc = OracleSim(m, dt, sub, (0.0, 0.0, 0.0))
    rng = np.random.default_rng(7)
    nb = 0 if m.root_fixed else 6
    for trial in range(4):
        root, dof = random_state(m, rng, z=5.0)
        root[7:] = 0; dof[:, 1] = 0
        tau = rng.normal(size=m.ndof) * 3
        qdd, ra, da = orc.forward_dynamics(root, dof, tau)
        acc = np.concatenate([(ra[7:13] - root[7:13]) / h, qdd]) if nb else qdd
        M = orc.mass_matrix(root[None], dof[None])[0]
        A = M + np.diag(np.r_[np.zeros(nb), h * m.damping[1:] + h * h * m.stiffness[1:]])
        rhs = np.r_[np.zeros(nb), np.clip(tau, -m.effort[1:], m.effort[1:]) - m.stiffness[1:] * dof[:, 0]]
        res = A @ acc - rhs
        assert np.abs(res).max() < 1e-9 * max(1.0, np.abs(rhs).max()), (name, trial, np.abs(res).max())


# ---------------------------------------------------------------------------------------------------------------
# the reference's indexing idiom for the operational-space controller (franka_cube_stack.py:388-394, 600-627) on the Franka itself
def test_franka_jacobian_is_indexed_by_joint_as_the_reference_does(reference_assets):
    """`hand_joint_index = gym.get_actor_joint_dict(env, franka)['panda_hand_joint']; j_eef = jacobian[:, hand_joint_index, :, :7]`:
    with one joint per non-root body the joint index addresses the hand body's row of the fixed-base Jacobian.  Checked on the
    Franka URDF (mesh collisions skipped with a warning: kinematics and inertias come from <inertial>): J_eef qd = the hand
    body's twist, and the task-space inertia (J M^-1 J^T)^-1 the controller forms is symmetric positive definite."""
    import warnings
    from isaacgymenvs_b200.importer.urdf import load_urdf
    from isaacgymenvs_b200.importer.model import BuildOptions, UnmodelledGeometryWarning
    from isaacgymenvs_b200.compat import gymapi
    with warnings.catch_warnings(record=True) as w:
        warnings.simplefilter("always")
        m = load_urdf(os.path.join(reference_assets, "urdf/franka_description/robots/franka_panda_gripper.urdf"), BuildOptions(fix_base_link=True))
    assert any(issubclass(x.category, UnmodelledGeometryWarning) for x in w) and len(m.unmodelled_geoms) == 11
    gym = gymapi.acquire_gym()
    asset = gymapi._Asset(m, gymapi.AssetOptions())
    jd = gym.get_asset_joint_dict(asset)
    assert gym.get_asset_joint_count(asset) == m.nb - 1 and jd["panda_joint1"] == 0
    hand = jd["panda_hand_joint"]
    assert m.body_names[hand + 1] == "panda_hand"
    orc = OracleSim(m, 0.0166, 2)
    root, dof = _states(m, 16, 8)
    J, M = orc.jacobian(root, dof), orc.mass_matrix(root, dof)
    Jh, Mh = _host_tensors(m, root, dof)                       # the kernel's arithmetic, on the CPU
    assert np.abs(Jh - J).max() < J_TOL and np.abs(Mh - M).max() < M_RTOL * np.abs(M).max()
    j_eef = J[:, hand, :, :7]                                   # (N, 6, 7) as franka_cube_stack.py:391
    tw = np.einsum("nrc,nc->nr", j_eef, dof[:, :7, 1])
    dof7 = dof.copy(); dof7[:, 7:, 1] = 0                       # the arm's seven joints are what moves the hand
    bs = orc.body_states(root, dof7)
    assert np.abs(tw[:, :3] - bs[:, hand + 1, 7:10]).max() < 1e-10 and np.abs(tw[:, 3:] - bs[:, hand + 1, 10:13]).max() < 1e-10
    mm = M[:, :7, :7]
    m_eef_inv = j_eef @ np.linalg.inv(mm) @ j_eef.transpose(0, 2, 1)           # :603-604; the controller inverts it (:605)
    assert np.abs(m_eef_inv - m_eef_inv.transpose(0, 2, 1)).max() < 1e-9 * np.abs(m_eef_inv).max()
    assert np.linalg.eigvalsh(0.5 * (m_eef_inv + m_eef_inv.transpose(0, 2, 1))).min() > 0 and np.isfinite(np.linalg.inv(m_eef_inv)).all()
