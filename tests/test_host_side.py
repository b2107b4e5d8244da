"""CPU-side checks that need no GPU: the C-ABI library builds, loads and exports every symbol
include/b200gym.h declares; the config loaders agree with the reference's YAML; importer
known-answers; the engine refuses to run without a CUDA device (no CPU fallback)."""
import ctypes
import os
import re
import numpy as np
import pytest

from tests.conftest import REFERENCE, ROOT


def test_library_builds_and_exports_the_declared_abi():
    from isaacgymenvs_b200 import build, engine
    path = build.build()
    lib = ctypes.CDLL(path)
    header = open(os.path.join(ROOT, "include", "b200gym.h")).read()
    declared = set(re.findall(r"\b(b2g_[a-z_]+)\s*\(", header))
    assert declared == set(engine.EXPORTS), declared ^ set(engine.EXPORTS)
    for sym in declared:
        assert hasattr(lib, sym), sym
    assert lib.b2g_version() == 4


def test_struct_layouts_match_header_sizes():
    """ctypes mirrors must have the size the C compiler gives the header's structs."""
    import subprocess, tempfile
    from isaacgymenvs_b200 import engine
    src = '#include "b200gym.h"\n#include <stdio.h>\nint main(){printf("%zu %zu %zu %zu %zu %zu\\n", sizeof(b2g_model), sizeof(b2g_sim_params), sizeof(b2g_task_params), sizeof(b2g_anymal_params), sizeof(b2g_model_ext), sizeof(b2g_hand_params));return 0;}\n'
    with tempfile.TemporaryDirectory() as d:
        open(os.path.join(d, "t.c"), "w").write(src)
        subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), "-o", os.path.join(d, "t"), os.path.join(d, "t.c")])
        sizes = [int(x) for x in subprocess.check_output([os.path.join(d, "t")]).split()]
    assert sizes == [ctypes.sizeof(engine.CModel), ctypes.sizeof(engine.CSimParams), ctypes.sizeof(engine.CTaskParams),
                     ctypes.sizeof(engine.CAnymalParams), ctypes.sizeof(engine.CModelExt), ctypes.sizeof(engine.CHandParams)]


def test_no_cpu_fallback():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    from isaacgymenvs_b200 import engine
    from isaacgymenvs_b200.assets import load_compiled
    with pytest.raises(engine.EngineError):
        engine.Sim(load_compiled("ant"), 4, 0.0166, 2, device="cuda:0")
    with pytest.raises(engine.EngineError):
        engine.Sim(load_compiled("ant"), 4, 0.0166, 2, device="cpu")


@pytest.mark.parametrize("task", ["Cartpole", "Ant", "Humanoid", "ShadowHand"])
def test_reference_yaml_loads_unmodified_and_matches_builtin(task, reference_cfg):
    """The built-in config against the reference's YAML as load_reference_cfg composes it (tests/golden/reference_cfg.json;
    where a reference checkout is present, also against a fresh load of its YAML)."""
    from isaacgymenvs_b200 import config
    ref = {"task": reference_cfg["task_cfg_num_envs_64"][task]}
    if os.path.isdir(REFERENCE):
        assert config.load_reference_cfg(os.path.join(REFERENCE, "isaacgymenvs", "cfg"), task, {"num_envs": 64})["task"] == ref["task"]
    own = config.builtin_cfg(task, {"num_envs": 64})

    def cmp(a, b, path=""):
        for k in b:
            assert k in a, path + k
            if isinstance(b[k], dict):
                cmp(a[k], b[k], path + k + ".")
            else:
                assert a[k] == b[k], (path + k, a[k], b[k])
    cmp(ref["task"], own["task"])
    assert ref["task"]["env"]["numEnvs"] == 64 and ref["task"]["sim"]["use_gpu_pipeline"] is True
    assert ref["task"]["sim"]["physx"]["num_threads"] == 4


def test_importer_known_answers_and_compiled_blobs_are_current(reference_assets):
    """SURVEY.md 8c importer known-answers (analytic, from the XML) + committed blobs == fresh import of the reference's
    robot descriptions (tests/golden/reference_assets.tar.xz)."""
    from isaacgymenvs_b200.importer.mjcf import load_mjcf
    from isaacgymenvs_b200.importer.urdf import load_urdf
    from isaacgymenvs_b200.importer.model import BuildOptions
    from isaacgymenvs_b200.assets import load_compiled
    from isaacgymenvs_b200.assets.compile_assets import SPECS
    ant = load_mjcf(os.path.join(reference_assets, "mjcf/nv_ant.xml"))
    assert abs(ant.mass[0] - 0.48388) < 1e-5 and abs(ant.mass[1] - 0.039158) < 1e-6 and abs(ant.mass[2] - 0.067592) < 1e-6
    assert abs(ant.total_mass() - 0.91088) < 1e-5
    assert ant.dof_names == ["hip_1", "ankle_1", "hip_2", "ankle_2", "hip_3", "ankle_3", "hip_4", "ankle_4"]
    assert np.allclose(np.degrees(ant.lower[1:3]), [-40, 30]) and np.allclose(ant.armature[1:], 0.01) and np.allclose(ant.damping[1:], 0.1)
    hum = load_mjcf(os.path.join(reference_assets, "mjcf/nv_humanoid.xml"))
    assert hum.nb == 16 and hum.ndof == 21 and hum.dof_names[:3] == ["abdomen_z", "abdomen_y", "abdomen_x"]
    assert hum.actuator_joint[:2] == ["abdomen_y", "abdomen_z"]
    cp = load_urdf(os.path.join(reference_assets, "urdf/cartpole.urdf"), BuildOptions(fix_base_link=True))
    assert cp.ndof == 2 and cp.jtype[1] == 1 and cp.jtype[2] == 0 and cp.limited[2] == 0 and abs(cp.lpos[2][0] - 0.12) < 1e-12
    any_ = load_urdf(os.path.join(reference_assets, "urdf/anymal_c/urdf/anymal_minimal.urdf"),
                     BuildOptions(collapse_fixed_joints=True, replace_cylinder_with_capsule=True))
    assert any_.nb == 13 and any_.ndof == 12 and len(any_.geom_type) == 9      # base + 4 x (knee, shank) ... feet
    for name, (rel, opts) in SPECS.items():
        path = os.path.join(reference_assets, rel)
        fresh = load_urdf(path, opts, name=name) if rel.endswith(".urdf") else load_mjcf(path, opts, name=name)
        blob = load_compiled(name)
        for f in ("parent", "jtype", "axis", "lpos", "mass", "com", "inertia", "lower", "upper", "cp_pos", "cp_radius", "limit_k"):
            assert np.allclose(getattr(fresh, f), getattr(blob, f)), (name, f)


@pytest.mark.parametrize("name", ["cartpole", "ant", "humanoid", "anymal", "shadow_hand"])
@pytest.mark.parametrize("lanes", [1, 2, 4, 8])
@pytest.mark.parametrize("compact", [False, True])
def test_slot_programs_are_consistent(name, lanes, compact):
    """The host-side list scheduler (b2g_plan = what b2g_create builds): every link is processed exactly once, after
    its parent; inertia hand-offs (carried in registers / parked in an accumulator / dropped under a fixed root) and
    the parents' child references agree."""
    from isaacgymenvs_b200 import engine
    from isaacgymenvs_b200.assets import load_compiled
    m = load_compiled(name)
    info, S = engine.plan(m, lanes, compact)
    ns, L = info["ns"], info["lanes"]
    assert L == lanes and 1 <= ns <= 24
    where = {}
    for s in range(24):
        for l in range(8):
            link = int(S[s, l, 0])
            if link >= 0:
                assert s < ns and l < L and link not in where and 1 <= link < m.nl
                where[link] = (l, s)
    assert sorted(where) == list(range(1, m.nl))
    crit = np.ones(m.nl, int)
    for i in range(m.nl - 1, 0, -1):
        crit[m.parent[i]] = max(crit[m.parent[i]], crit[i] + 1)
    assert ns >= crit[0] - 1                                        # never shorter than the longest chain below the root
    if lanes == 1:
        assert ns == m.nl - 1 and info["cross_lane"] == 0
    parked = {}
    cross = 0
    for link, (l, s) in where.items():
        rec = S[s, l]
        p = int(m.parent[link])
        if p == 0:
            assert rec[1] == 0
            if rec[2] != -1:
                assert s > 0 and (rec[2] == info["root_acc"] or (rec[2] == -2 and compact and m.root_fixed))
            else:
                assert s == 0
        else:
            pl, ps = where[p]
            assert ps < s and rec[1] == ((pl << 8) | (ps + 1))
            cross |= int(pl != l)
            if pl == l and ps == s - 1:
                assert rec[2] == -1
            else:
                assert rec[2] >= 0 and rec[2] < info["nacc"]
                parked[link] = (l, int(rec[2]))
    assert cross == info["cross_lane"]
    # every parked inertia is collected exactly once, by its parent
    seen = {}
    for link, (l, s) in where.items():
        refs = [int(c) for c in S[s, l, 4:8] if c >= 0]
        assert (int(S[s, l, 3]) & 1) == int(len(refs) > 0)
        for r in refs:
            seen[r] = seen.get(r, 0) + 1
            kids = [k for k, v in parked.items() if int(m.parent[k]) == link and ((v[0] << 8) | v[1]) == r or (compact and int(m.parent[k]) == link and v[1] == (r & 255))]
            assert len(kids) == 1, (link, r, kids)
    assert sum(seen.values()) == len(parked) and all(v == 1 for v in seen.values())
    if compact:                                                     # env-wide ids are unique
        ids = [v[1] for v in parked.values()]
        assert len(set(ids)) == len(ids)


@pytest.mark.parametrize("workload", ["ant", "shadow_hand"])
def test_bench_reference_arm_prints_the_contract_line(workload):
    """`bench.py --impl reference` (the CPU port of the path on host cores) runs without a GPU and prints ONE JSON line
    with the keys the driver reads."""
    import json, subprocess, sys
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", workload,
                          "--steps", "2", "--warmup", "1", "--gpus", "1"], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
              "dtype", "data", "config", "impl", "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["impl"] == "reference" and d["unit"] == "env-steps/s" and d["value"] > 0 and d["higher_is_better"] is True
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["vs_baseline"] is None and "workload" in d["config"]


def test_bench_dump_outputs_writes_what_step_returned(tmp_path, monkeypatch):
    """bench.py --dump-outputs: one float32 / float64 .npy per array VecTask.step() returns; above the size limit every per-env
    array keeps the same seeded sample of envs, whose indices are written beside them."""
    import importlib.util, torch
    spec = importlib.util.spec_from_file_location("b2g_bench", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec); spec.loader.exec_module(bench)
    n = 1000
    g = torch.Generator().manual_seed(1)
    result = ({"obs": torch.rand(n, 60, generator=g)}, torch.rand(n, generator=g, dtype=torch.float64), torch.randint(0, 2, (n,), generator=g),
              {"time_outs": torch.rand(n, generator=g) > 0.5, "consecutive_successes": torch.tensor(1.5), "episode": 3})
    outs = bench.step_outputs(result)
    assert sorted(outs) == ["consecutive_successes", "obs", "reset", "rew", "time_outs"]
    assert outs["rew"].dtype == np.float64 and all(outs[k].dtype == np.float32 for k in ("obs", "reset", "time_outs", "consecutive_successes"))
    assert np.array_equal(outs["reset"], result[2].numpy()) and np.array_equal(outs["obs"], result[0]["obs"].numpy())
    bench.dump_outputs(outs, str(tmp_path / "whole"))
    for k, a in outs.items():
        assert np.array_equal(np.load(tmp_path / "whole" / f"{k}.npy"), a)
    assert not (tmp_path / "whole" / "sample_envs.npy").exists()
    monkeypatch.setattr(bench, "DUMP_LIMIT_BYTES", 100_000)
    for d in ("s1", "s2"):
        bench.dump_outputs(dict(outs), str(tmp_path / d))
    got = {k: np.load(tmp_path / "s1" / f"{k}.npy") for k in list(outs) + ["sample_envs"]}
    rows = got["sample_envs"].astype(np.int64)
    assert got["sample_envs"].dtype == np.float64 and 0 < len(rows) < n and sum(a.nbytes for a in got.values()) <= 100_000
    for k in ("obs", "rew", "reset", "time_outs"):
        assert np.array_equal(got[k], outs[k][rows])
        assert np.array_equal(np.load(tmp_path / "s2" / f"{k}.npy"), got[k])
    assert got["consecutive_successes"] == np.float32(1.5)


@pytest.mark.gpu
def test_bench_dump_outputs_of_the_gpu_path(tmp_path):
    """`bench.py --dump-outputs DIR` on the GPU: the last timed step's observation / reward / reset / time-out arrays land in DIR
    and the JSON line reports the requested step count."""
    import json, subprocess, sys
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", "3", "--warmup", "1", "--num-envs", "512",
                          "--sets", "2", "--no-cpu-baseline", "--no-rollout", "--dump-outputs", str(tmp_path / "out")],
                         capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    d = json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][0])
    assert d["steps"] == 3
    got = {f[:-4]: np.load(tmp_path / "out" / f) for f in os.listdir(tmp_path / "out")}
    assert {"obs", "rew", "reset", "time_outs"} <= set(got) and got["obs"].shape == (512, 60) and got["rew"].shape == (512,)
    assert all(a.dtype in (np.float32, np.float64) and np.isfinite(a).all() for a in got.values())


def test_bench_reference_arm_other_ranks_exit_quietly():
    import subprocess, sys
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--gpus", "2"],
                         capture_output=True, text=True, timeout=120, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_domain_randomisation_noise_matches_reference():
    """isaacgymenvs_b200.utils.dr.NoiseModel against the lambdas the reference's own VecTask.apply_randomizations
    installs (tests/golden/make_golden_dr.py): same torch seed -> same numbers, for gaussian / uniform, additive /
    scaling, linear / constant / no schedule, first call (draws the correlated sample) and second call (re-uses it)."""
    import sys, torch
    from isaacgymenvs_b200.utils.dr import NoiseModel, Randomizer
    sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
    import make_golden_dr as G
    gold = np.load(os.path.join(ROOT, "tests", "golden", "dr_noise.npz"))
    checked = 0
    for cname, params in G.CASES.items():
        for frame in G.FRAMES:
            for key in ("observations", "actions"):
                if key not in params:
                    continue
                x = torch.tensor(gold[f"x_{key}"])
                nm = NoiseModel(params[key], frame)
                torch.manual_seed(1000 + frame)
                y1 = nm(x.clone()); y2 = nm(x.clone())
                np.testing.assert_allclose(y1.numpy(), gold[f"{cname}_{frame}_{key}_1"], rtol=0, atol=1e-7)
                np.testing.assert_allclose(y2.numpy(), gold[f"{cname}_{frame}_{key}_2"], rtol=0, atol=1e-7)
                checked += 1
    assert checked == 25
    # frequency gating (vec_task.py:619-640): first call always, then every `frequency` frames
    r = Randomizer({"frequency": 10, "observations": G.CASES["uniform_scale"]["observations"]})
    assert r.update(0) and not r.update(5) and r.update(10) and not r.update(19) and r.update(20)
    with pytest.raises(NotImplementedError):
        Randomizer({"frequency": 1, "sim_params": {}})


def test_self_collision_request_is_never_silent():
    """Self-collision (create_actor collision_filter 0 / -1: humanoid.py:194, anymal_terrain.py:282, shadow_hand.py:359) is not
    modelled; asking for it must be audible: one UnmodelledPhysicsWarning per actor kind."""
    import warnings
    from isaacgymenvs_b200 import engine
    engine._warned.discard("probe")
    with warnings.catch_warnings(record=True) as rec:
        warnings.simplefilter("always")
        engine.warn_self_collision("probe", "create_actor(..., 0, 0)")
        engine.warn_self_collision("probe", "create_actor(..., 0, 0)")
    assert len(rec) == 1 and issubclass(rec[0].category, engine.UnmodelledPhysicsWarning) and "self-collision" in str(rec[0].message)


# ---------------------------------------------------------------------------------------------
# general triangle-mesh terrain for gym.add_triangle_mesh (SURVEY 8f rank 4): sampled onto the engine's height field
def test_trimesh_terrain_is_sampled_back_onto_its_height_field():
    from isaacgymenvs_b200 import terrain as T
    rng = np.random.default_rng(0)
    hf = (rng.integers(-40, 60, size=(23, 31))).astype(np.int16)
    hs, vs = 0.25, 0.005
    v, t = T.convert_heightfield_to_trimesh(hf, hs, vs, None)
    # strip the tag: what a caller with its own mesh would pass (flat arrays, anymal_terrain.py:206)
    v0, t0 = np.array(v, dtype=np.float32).flatten(order="C"), np.array(t, dtype=np.uint32).flatten(order="C")
    out = T.trimesh_to_heightfield(v0, t0)
    assert out["horizontal_scale"] == pytest.approx(hs) and out["offset"] == (0.0, 0.0)
    rec = out["height_field"].astype(np.float64) * out["vertical_scale"]
    assert rec.shape == hf.shape and np.abs(rec - hf * vs).max() <= 0.5 * out["vertical_scale"] + 1e-7
    # a coarser grid over a tilted plane made of two triangles, not aligned with the origin
    P = np.array([[1.0, -2.0, 0.1], [5.0, -2.0, 0.5], [5.0, 1.0, 0.8], [1.0, 1.0, 0.4]])
    tri = np.array([[0, 1, 2], [0, 2, 3]])
    o2 = T.trimesh_to_heightfield(P, tri, horizontal_scale=0.5)
    gx = o2["offset"][0] + 0.5 * np.arange(o2["height_field"].shape[0]); gy = o2["offset"][1] + 0.5 * np.arange(o2["height_field"].shape[1])
    want = 0.1 + 0.1 * (gx[:, None] - 1.0) + 0.1 * (gy[None, :] + 2.0)
    assert np.abs(o2["height_field"] * o2["vertical_scale"] - want).max() <= 0.5 * o2["vertical_scale"] + 1e-9
    # a box on a floor: the upper surface wins above the box, its vertical walls carry no height of their own
    fl = np.array([[0, 0, 0], [4, 0, 0], [4, 4, 0], [0, 4, 0]], float); bx = np.array([[1, 1, 0.5], [3, 1, 0.5], [3, 3, 0.5], [1, 3, 0.5]], float)
    walls = np.array([[1, 1, 0], [3, 1, 0], [3, 1, 0.5], [1, 1, 0.5]], float)
    V = np.concatenate([fl, bx, walls]); F = np.array([[0, 1, 2], [0, 2, 3], [4, 5, 6], [4, 6, 7], [8, 9, 10], [8, 10, 11]])
    o3 = T.trimesh_to_heightfield(V, F, horizontal_scale=0.5)
    h3 = o3["height_field"] * o3["vertical_scale"]
    assert h3.shape == (9, 9) and h3[4, 4] == pytest.approx(0.5, abs=1e-3) and h3[0, 0] == 0.0 and h3[2, 2] == pytest.approx(0.5, abs=1e-3) and h3[1, 4] == 0.0
    with pytest.raises(ValueError):
        T.trimesh_to_heightfield(V, np.array([[0, 1, 99]]))


def test_compat_add_triangle_mesh_accepts_an_untagged_mesh():
    from isaacgymenvs_b200.compat import gymapi
    from isaacgymenvs_b200 import terrain as T
    gym = gymapi.acquire_gym()
    sp = gymapi.SimParams(); sp.dt = 0.005; sp.substeps = 1
    sim = gym.create_sim(0, -1, gymapi.SIM_PHYSX, sp)
    hf = (np.arange(12 * 9).reshape(12, 9) % 7).astype(np.int16)
    v, t = T.convert_heightfield_to_trimesh(hf, 0.1, 0.005, None)
    tp = gymapi.TriangleMeshParams()
    tp.nb_vertices, tp.nb_triangles = v.shape[0], t.shape[0]
    tp.transform.p.x, tp.transform.p.y, tp.transform.p.z = -2.0, -3.0, 0.0
    tp.static_friction = tp.dynamic_friction = 0.9
    gym.add_triangle_mesh(sim, np.array(v).flatten(), np.array(t).flatten(), tp)           # np.array(): the tag is gone
    tr = sim.terrain
    assert tr["origin"] == (-2.0, -3.0) and tr["friction"] == pytest.approx(0.9) and tr["height_field"].shape == (12, 9)
    assert np.abs(tr["height_field"] * tr["vertical_scale"] - hf * 0.005).max() <= 0.5 * tr["vertical_scale"] + 1e-7
    tp.nb_vertices = 5
    with pytest.raises(ValueError):
        gym.add_triangle_mesh(sim, np.array(v).flatten(), np.array(t).flatten(), tp)


# ---------------------------------------------------------------------------------------------
# train.py: the reference launcher's override syntax over the demonstration learner
def test_train_launcher_maps_reference_overrides():
    import importlib.util
    spec = importlib.util.spec_from_file_location("b2g_train", os.path.join(ROOT, "train.py"))
    tr = importlib.util.module_from_spec(spec); spec.loader.exec_module(tr)
    a = tr.to_ppo_argv(tr.parse_overrides(["task=ShadowHand", "headless=True", "num_envs=8192", "max_iterations=300", "seed=7",
                                           "task.env.objectType=pen", "task.env.forceScale=1.0"]))
    get = lambda k: a[a.index(k) + 1]
    assert get("--task") == "ShadowHand" and get("--num-envs") == "8192" and get("--epochs") == "300" and get("--seed") == "7"
    assert get("--units") == "512,512,256,128" and float(get("--kl-threshold")) == 0.016 and get("--horizon") == "8"
    assert get("--env") == "objectType=pen,forceScale=1.0"
    b = tr.to_ppo_argv(tr.parse_overrides(["task=Humanoid", "task.env.selfCollision=True"]))
    assert "--self-collision" in b and "--env" not in b and b[b.index("--epochs") + 1] == "1000"
    for bad in (["task=FrankaCabinet"], ["task=Ant", "train.params.config.gamma=0.9"], ["task=Ant", "test=True"], ["Ant"]):
        with pytest.raises(SystemExit):
            tr.to_ppo_argv(tr.parse_overrides(bad))


def test_train_launcher_hyperparameters_are_the_reference_yaml(reference_cfg):
    """train.py's PPO table against the values of the reference's train / task YAML (tests/golden/reference_cfg.json)."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("b2g_train", os.path.join(ROOT, "train.py"))
    tr = importlib.util.module_from_spec(spec); spec.loader.exec_module(tr)
    assert sorted(reference_cfg["ppo"]) == sorted(tr.PPO)
    for task, hp in tr.PPO.items():
        c = reference_cfg["ppo"][task]
        assert c["units"] == hp["units"] and float(c["learning_rate"]) == hp["lr"] and c["horizon_length"] == hp["horizon"]
        assert c["minibatch_size"] == hp["minibatch"] and c["mini_epochs"] == hp["mini_epochs"] and c["critic_coef"] == hp["critic_coef"]
        assert c["kl_threshold"] == hp["kl"] and c["scale_value"] == hp["rew_scale"] and float(c["bounds_loss_coef"]) == hp["bounds"]
        assert str(hp["epochs"]) in c["max_epochs"] and c["gamma"] == 0.99 and c["tau"] == 0.95 and c["e_clip"] == 0.2
        assert str(hp["num_envs"]) in c["num_envs"]


# ---------------------------------------------------------------------------------------------
# collision meshes: mass properties of the enclosed volume (importer/mesh.py), skipped contact announced
def test_mesh_mass_properties_are_those_of_the_enclosed_solid(tmp_path):
    from isaacgymenvs_b200.importer.mesh import load_obj, mass_properties
    from isaacgymenvs_b200.importer import rot
    h, c0 = np.array([1.0, 2.0, 3.0]), np.array([0.3, -0.2, 0.5])
    R = rot.quat_to_mat(np.array([0.2, -0.1, 0.3, 0.9]) / np.linalg.norm([0.2, -0.1, 0.3, 0.9]))
    corners = np.array([[sx, sy, sz] for sx in (-1, 1) for sy in (-1, 1) for sz in (-1, 1)], float) * h
    ix = lambda sx, sy, sz: (0 if sx < 0 else 4) + (0 if sy < 0 else 2) + (0 if sz < 0 else 1)
    quads = [[ix(1, -1, -1), ix(1, 1, -1), ix(1, 1, 1), ix(1, -1, 1)], [ix(-1, -1, -1), ix(-1, -1, 1), ix(-1, 1, 1), ix(-1, 1, -1)],
             [ix(-1, 1, -1), ix(-1, 1, 1), ix(1, 1, 1), ix(1, 1, -1)], [ix(-1, -1, -1), ix(1, -1, -1), ix(1, -1, 1), ix(-1, -1, 1)],
             [ix(-1, -1, 1), ix(1, -1, 1), ix(1, 1, 1), ix(-1, 1, 1)], [ix(-1, -1, -1), ix(-1, 1, -1), ix(1, 1, -1), ix(1, -1, -1)]]
    V = corners @ R.T + c0
    p = tmp_path / "box.obj"
    with open(p, "w") as f:                                   # quads, 1-based, with normal indices: what Meshlab writes
        f.write("# test\n" + "".join(f"v {x} {y} {z}\n" for x, y, z in V) + "".join("f " + " ".join(f"{i + 1}//{i + 1}" for i in q) + "\n" for q in quads))
    Vr, F = load_obj(str(p))
    assert F.shape == (12, 3)
    vol, com, I = mass_properties(Vr, F)
    Ibox = 48.0 / 12.0 * np.diag([16 + 36, 4 + 36, 4 + 16.0])
    assert vol == pytest.approx(48.0, rel=1e-12) and np.allclose(com, c0, atol=1e-12) and np.allclose(I, R @ Ibox @ R.T, atol=1e-9)
    vol2, com2, I2 = mass_properties(Vr, F[:, ::-1])          # inward-facing triangles: same solid
    assert vol2 == pytest.approx(48.0) and np.allclose(com2, c0) and np.allclose(I2, I)
    with pytest.raises(ValueError):
        mass_properties(np.zeros((3, 3)), np.array([[0, 1, 2]]))


def test_franka_links_get_their_mass_from_the_collision_meshes(reference_assets):
    """franka_panda_gripper.urdf has no <inertial>: density x mesh volume (AssetOptions.density 1000) must give a ~20 kg arm, and
    the skipped mesh CONTACT is announced, not silent."""
    import warnings
    from isaacgymenvs_b200.importer.urdf import load_urdf
    from isaacgymenvs_b200.importer.model import BuildOptions, UnmodelledGeometryWarning
    with warnings.catch_warnings(record=True) as w:
        warnings.simplefilter("always")
        m = load_urdf(os.path.join(reference_assets, "urdf/franka_description/robots/franka_panda_gripper.urdf"), BuildOptions(fix_base_link=True))
    assert sum(issubclass(x.category, UnmodelledGeometryWarning) for x in w) == 1
    assert 15.0 < m.total_mass() < 25.0 and (m.mass[:8] > 1.0).all() and (m.inertia[1:8, :3] > 1e-3).all()
    assert m.body_joint_names[8] == "panda_hand_joint" and m.body_names[8] == "panda_hand" and m.ndof == 9


def test_compiled_models_carry_joint_names_and_announce_skipped_meshes():
    """what the GPU box sees (no XML there): the blobs know their joint names (gym.get_actor_joint_dict) and the fallback loader
    repeats the importer's warning about collision meshes without a contact model"""
    import warnings
    from isaacgymenvs_b200.assets import load_compiled, load_asset_file, KNOWN
    from isaacgymenvs_b200.importer.model import BuildOptions, UnmodelledGeometryWarning
    from isaacgymenvs_b200.compat import gymapi
    gym = gymapi.acquire_gym()
    for name in set(KNOWN.values()):
        m = load_compiled(name)
        assert len(m.body_joint_names) == m.nb and m.body_joint_names[0] == ""
        jd = gym.get_asset_joint_dict(gymapi._Asset(m, gymapi.AssetOptions()))
        assert all(m.body_joint_names[i + 1] == n for n, i in jd.items())
    assert gym.get_asset_joint_dict(gymapi._Asset(load_compiled("franka"), gymapi.AssetOptions()))["panda_hand_joint"] == 7
    with warnings.catch_warnings(record=True) as w:
        warnings.simplefilter("always")
        load_asset_file("/no/such/checkout/assets", "urdf/franka_description/robots/franka_panda_gripper.urdf", BuildOptions(fix_base_link=True))
        load_asset_file("/no/such/checkout/assets", "mjcf/nv_ant.xml", BuildOptions())
    hits = [x for x in w if issubclass(x.category, UnmodelledGeometryWarning)]
    assert len(hits) == 1 and "franka" in str(hits[0].message)
