"""Generate the fixtures of the boundary tests (tests/test_host.py, tests/test_reference_callers.py) by running the reference's
own code once, so that the tests themselves need nothing outside this repository.

Run where the reference checkout exists (V2P_REFERENCE, see _refenv.py):  python tests/golden/make_golden_host.py

Fixtures
  poselib_quat.npz                    poselib.core.rotation3d quat_mul / quat_conjugate / quat_from_angle_axis / quat_rotate on
                                      seeded inputs
  amass_asset/                        the reference's MJCF asset smpl_mesh_humanoid_amass_v1 with its STL meshes (data, same
                                      relative layout), input of model_compiler.compile_mjcf
  ref_motion_lib.pth                  `torch.save` of a reference MotionLib (utils/motion_lib.py) built from a small synthetic library
  ref_callers.json                    what the reference's VecTaskPythonWrapper + RLGPUEnv touch on a task object, and the calls
                                      utils/config.py (get_args / load_cfg / parse_sim_params) makes into the isaacgym shim
"""
import json
import os
import shutil
import subprocess
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, HERE)
sys.path.insert(0, REPO)
import _refenv  # noqa: E402

REF = _refenv.REF


def poselib_quat():
    sys.path.insert(0, os.path.join(REF, "poselib"))
    from poselib.core import rotation3d as P
    g = torch.Generator().manual_seed(0)
    a = torch.nn.functional.normalize(torch.randn(64, 4, generator=g), dim=-1)
    b = torch.nn.functional.normalize(torch.randn(64, 4, generator=g), dim=-1)
    v = torch.randn(64, 3, generator=g)
    ang = torch.rand(64, generator=g) * 6 - 3
    np.savez_compressed(os.path.join(HERE, "poselib_quat.npz"), a=a.numpy(), b=b.numpy(), v=v.numpy(), ang=ang.numpy(),
                        quat_mul=P.quat_mul(a, b).numpy(), quat_conjugate=P.quat_conjugate(a).numpy(),
                        quat_from_angle_axis=P.quat_from_angle_axis(ang, v).numpy(), quat_rotate=P.quat_rotate(a, v).numpy())


def mjcf_asset():
    src, dst = os.path.join(REF, "embodied_pose", "data", "assets"), os.path.join(HERE, "amass_asset")
    xml = os.path.join("mjcf", "smpl_mesh_humanoid_amass_v1.xml")
    os.makedirs(os.path.join(dst, "mjcf"), exist_ok=True)
    shutil.copyfile(os.path.join(src, xml), os.path.join(dst, xml))
    meshes = os.path.join("mesh", "smpl", "5117b308-a58e-4020-9d6b-4dd1930a10f6", "geom")
    shutil.copytree(os.path.join(src, meshes), os.path.join(dst, meshes), copy_function=shutil.copyfile, dirs_exist_ok=True)


def ref_motion_lib():
    code = r'''
import sys
sys.path.insert(0, %(here)r); sys.path.insert(0, %(repo)r)
import torch
import numpy as np
import make_golden as G
from vid2player3d_b200 import model_compiler, motion_lib
model = model_compiler.load_compiled("smpl_mesh_humanoid_amass_v1")
flat = motion_lib.synthetic(model, num_motions=3, num_frames=12, seed=11, sigma=0.08, ragged=True)
flat.min_verts_h = np.linspace(-0.02, 0.03, 3).astype(np.float32)
flat.motion_bodies = np.random.default_rng(5).normal(size=(3, 11)).astype(np.float32)
names = [str(n) for n in model["body_names"]]
key = [names.index(n) for n in ["R_Ankle", "L_Ankle", "L_Hand", "R_Hand"]]
torch.save(G.make_ref_motion_lib(flat, key, model["dof_body_ids"]), %(out)r)
''' % {"here": HERE, "repo": REPO, "out": os.path.join(HERE, "ref_motion_lib.pth")}
    subprocess.check_call([sys.executable, "-c", code])


CALLERS = r'''
import json, os, sys
sys.path.insert(0, %(here)r); sys.path.insert(0, %(repo)r)
import _refenv
_refenv.setup("embodied_pose")
import torch, types
import numpy as _np
if not hasattr(_np, 'Inf'):
    _np.Inf = _np.inf          # the reference targets numpy < 2 (vec_task.py:28-30)
for _pkg in ("agents", "players", "models", "learning"):          # the reference's top-level packages (no __init__.py): make sure they
    _m = types.ModuleType(_pkg)                                  # are not shadowed by same-named site-packages
    _m.__path__ = [os.path.join(_refenv.REF, "embodied_pose", _pkg)]
    sys.modules[_pkg] = _m
import rl_games.common                                             # mocked (rl_games 1.1.4 is not installed); RLGPUEnv needs a real base class
_ve = types.ModuleType("rl_games.common.vecenv")
class _IVecEnv: pass
_ve.IVecEnv, _ve.register = _IVecEnv, (lambda *a, **k: None)
rl_games.common.vecenv = sys.modules["rl_games.common.vecenv"] = _ve
from env.tasks.vec_task_wrappers import VecTaskPythonWrapper      # the reference's classes, unchanged
import run as ref_run

def make_rlgpu(env):
    e = ref_run.RLGPUEnv.__new__(ref_run.RLGPUEnv)     # __init__ only looks the env creator up in rl_games' registry
    e.env, e.use_global_obs, e.full_state = env, env.num_states > 0, {}
    e.full_state["obs"] = e.reset()
    return e

class Recorder:
    """stand-in with the buffer contract of BaseTask (base_task.py:62-74); records what the reference code touches"""
    def __init__(self):
        object.__setattr__(self, "touched", set())
        d = dict(num_envs=6, num_obs=461, num_states=0, num_actions=75, obs_buf=torch.randn(6, 461) * 9, states_buf=torch.zeros(6, 0),
                 rew_buf=torch.rand(6), reset_buf=torch.zeros(6, dtype=torch.long), progress_buf=torch.zeros(6, dtype=torch.long),
                 extras={"terminate": torch.zeros(6, dtype=torch.long)}, steps=[])
        object.__setattr__(self, "d", d)
    def __getattr__(self, k):
        self.touched.add(k)
        if k == "step":
            return lambda a: self.d["steps"].append(tuple(a.shape))
        if k == "reset":
            return lambda ids=None: self.d["steps"].append(("reset", None if ids is None else len(ids)))
        return self.d[k]

t = Recorder()
vec = VecTaskPythonWrapper(t, "cpu", 5.0, 1.0)
env = make_rlgpu(vec)
obs = env.reset()
for _ in range(3):
    obs, rew, done, info = env.step(torch.randn(6, 75) * 3)
env.reset(torch.tensor([1, 4]))
info_d = env.get_env_info()
callers = {"touched": sorted(t.touched), "steps": t.d["steps"], "obs_max": float(obs.abs().max()),
           "n_agents": env.get_number_of_agents(), "info_keys": sorted(info_d)}

# utils/config.py against the shim: record every call it makes into isaacgym.gymutil, and the SimParams it ends with
from isaacgym import gymapi, gymutil
calls = {}
_pa, _psc = gymutil.parse_arguments, gymutil.parse_sim_config
def parse_arguments(**kw):
    calls["parse_arguments"] = {"kwargs": {k: v for k, v in kw.items() if k != "custom_parameters"},
                                "custom_parameters": [{k: (v.__name__ if isinstance(v, type) else v) for k, v in p.items()}
                                                      for p in kw.get("custom_parameters", [])], "argv": list(sys.argv[1:])}
    args = _pa(**kw)
    calls["parse_arguments"]["result"] = {k: v for k, v in vars(args).items()}
    return args
def parse_sim_config(sim_cfg, sim_options):
    calls["parse_sim_config"] = {"sim_cfg": sim_cfg}
    return _psc(sim_cfg, sim_options)
gymutil.parse_arguments, gymutil.parse_sim_config = parse_arguments, parse_sim_config
sys.argv = ["run.py", "--cfg", "amass_im", "--headless", "--num_envs", "64"]
from utils.config import get_args, load_cfg, parse_sim_params
os.chdir(_refenv.REF)
args = get_args()
cfg, cfg_train = load_cfg(args)
sp = parse_sim_params(args, cfg, cfg_train)
fields = lambda o: {k: (list(v) if isinstance(v, gymapi.Vec3) else v) for k, v in vars(o).items() if k not in ("physx", "flex")}
calls["sim_params"] = dict(fields(sp), physx=fields(sp.physx), flex=fields(sp.flex))
calls["cfg"] = {"numEnvs": cfg["env"]["numEnvs"], "name": cfg["name"]}
print(json.dumps({"callers": callers, "config": calls}))
'''


def ref_callers():
    r = subprocess.run([sys.executable, "-c", CALLERS % {"here": HERE, "repo": REPO}], capture_output=True, text=True, check=True)
    out = json.loads(r.stdout.strip().splitlines()[-1])
    with open(os.path.join(HERE, "ref_callers.json"), "w") as f:
        json.dump(out, f, indent=1, sort_keys=True)
        f.write("\n")


if __name__ == "__main__":
    assert _refenv.available(), f"reference checkout not found at {REF} (set V2P_REFERENCE)"
    poselib_quat()
    mjcf_asset()
    ref_motion_lib()
    ref_callers()
