"""Golden data for the host-side tests that compare with the reference's configuration and robot descriptions:
    python tests/golden/make_golden_reference_data.py <IsaacGymEnvs checkout>
Writes
  reference_cfg.json  -- the task configs as config.load_reference_cfg composes them from the checkout's YAML (num_envs=64),
                         and the PPO hyper-parameters / env counts of the train and task YAML that train.py restates;
  reference_assets.tar.xz -- the robot descriptions (MJCF / URDF, the Franka's collision meshes) the importer reads for every
                         compiled model (isaacgymenvs_b200/assets/compile_assets.py SPECS), with their licenses.
Both are reproducible byte for byte from the same checkout."""
import importlib.util
import io
import json
import os
import sys
import tarfile

import yaml

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
OUT = os.path.dirname(os.path.abspath(__file__))

CFG_TASKS = ["Cartpole", "Ant", "Humanoid", "ShadowHand"]
ASSETS = ["mjcf/nv_ant.xml", "mjcf/nv_humanoid.xml", "urdf/cartpole.urdf", "urdf/anymal_c/urdf/anymal_minimal.urdf",
          "urdf/objects/cube_multicolor.urdf", "urdf/franka_description/robots/franka_panda_gripper.urdf"] + \
         [f"mjcf/open_ai_assets/hand/{f}.xml" for f in ("shadow_hand", "shared", "shared_asset", "robot", "egg", "pen")] + \
         [f"urdf/franka_description/meshes/collision/{f}.obj" for f in ("finger", "hand") + tuple(f"link{i}" for i in range(8))] + \
         [f"licenses/{f}-LICENSE.txt" for f in ("ant", "anymal_c", "cartpole", "franka", "humanoid", "open_ai_assets")]


def ppo_values(ref):
    spec = importlib.util.spec_from_file_location("b2g_train", os.path.join(ROOT, "train.py"))
    tr = importlib.util.module_from_spec(spec); spec.loader.exec_module(tr)
    out = {}
    for task in tr.PPO:
        with open(os.path.join(ref, "isaacgymenvs", "cfg", "train", task + "PPO.yaml")) as f:
            d = yaml.safe_load(f)
        c, n = d["params"]["config"], d["params"]["network"]
        with open(os.path.join(ref, "isaacgymenvs", "cfg", "task", task + ".yaml")) as f:
            t = yaml.safe_load(f)
        out[task] = {"units": n["mlp"]["units"], "num_envs": str(t["env"]["numEnvs"]), "scale_value": c["reward_shaper"]["scale_value"],
                     **{k: c[k] for k in ("learning_rate", "horizon_length", "minibatch_size", "mini_epochs", "critic_coef",
                                          "kl_threshold", "bounds_loss_coef", "max_epochs", "gamma", "tau", "e_clip")}}
    return out


def main(ref):
    from isaacgymenvs_b200 import config
    cfg = {task: config.load_reference_cfg(os.path.join(ref, "isaacgymenvs", "cfg"), task, {"num_envs": 64})["task"] for task in CFG_TASKS}
    with open(os.path.join(OUT, "reference_cfg.json"), "w") as f:
        json.dump({"task_cfg_num_envs_64": cfg, "ppo": ppo_values(ref)}, f, indent=1, sort_keys=True)
        f.write("\n")
    buf = io.BytesIO()
    with tarfile.open(fileobj=buf, mode="w", format=tarfile.USTAR_FORMAT) as tar:
        for rel in sorted(ASSETS):
            with open(os.path.join(ref, "assets", rel), "rb") as f:
                data = f.read()
            info = tarfile.TarInfo(rel)
            info.size, info.mode, info.mtime = len(data), 0o644, 0
            tar.addfile(info, io.BytesIO(data))
    import lzma
    with open(os.path.join(OUT, "reference_assets.tar.xz"), "wb") as f:
        f.write(lzma.compress(buf.getvalue(), preset=9 | lzma.PRESET_EXTREME))


if __name__ == "__main__":
    main(sys.argv[1])
