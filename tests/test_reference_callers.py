"""Caller-side proof of the boundary (SURVEY.md 8b, VERDICT r1 item 6): the REFERENCE's own rl_games-facing code -
`VecTaskPythonWrapper` (embodied_pose/env/tasks/vec_task.py:16-63,120-138, vec_task_wrappers.py:22-28) and `RLGPUEnv.step/reset`
(embodied_pose/run.py:93-137) - driven over a task object.

The reference classes were run once over a recording stand-in with CPU buffers (tests/golden/make_golden_host.py); what they
touched on the task and what they did with it is stored in tests/golden/ref_callers.json.
  * CPU part: every attribute / method the reference's callers touch must be provided by the B200 task classes.
  * GPU part: `vid2player3d_b200.tasks.HumanoidSMPLIM` driven for 32 steps the way those callers drive it (clipped actions,
    clipped observations, reset of the finished envs), every touched attribute present on the live task, and
    `b200env_obs_imitation` on the live GPU buffers matching the numpy port of the reference's
    `compute_humanoid_observations_imitation` (oracle/ref_port.py, pinned to the reference by tests/test_oracle_golden.py)."""
import json
import os
import re

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CALLERS = os.path.join(ROOT, "tests", "golden", "ref_callers.json")


def _recorded():
    with open(CALLERS) as f:
        return json.load(f)["callers"]


def _provided_names():
    """attributes the B200 task classes define: class members + every `self.<name> =` of their sources (no CUDA needed)"""
    from vid2player3d_b200.tasks import base_task, humanoid_smpl_im
    names = set(dir(humanoid_smpl_im.HumanoidSMPLIM))
    for mod in (base_task, humanoid_smpl_im):
        names |= set(re.findall(r"self\.([A-Za-z_][A-Za-z_0-9]*)\s*(?:,\s*self\.[A-Za-z_0-9]+\s*)*=", open(mod.__file__).read()))
        names |= set(re.findall(r"self\.([A-Za-z_][A-Za-z_0-9]*)", open(mod.__file__).read()))
    return names


def test_reference_vec_task_and_rlgpu_env_touch_only_what_the_b200_task_provides():
    out = _recorded()
    provided = _provided_names()
    missing = [n for n in out["touched"] if n not in provided]
    assert not missing, f"the reference's callers touch task attributes the B200 task does not define: {missing}"
    assert out["obs_max"] <= 5.0 and out["n_agents"] == 1 and out["info_keys"] == ["action_space", "observation_space"]
    assert out["steps"][0] == ["reset", None] and out["steps"][-1] == ["reset", 2] and out["steps"].count([6, 75]) == 3


@pytest.mark.gpu
def test_reference_callers_drive_the_b200_task_on_the_gpu():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    from oracle import ref_port as R
    from vid2player3d_b200 import model_compiler, motion_lib
    from vid2player3d_b200.configs import SIM_PARAMS, im_cfg
    from vid2player3d_b200.tasks import HumanoidSMPLIM
    model = model_compiler.load_compiled("smpl_mesh_humanoid_amass_v1")
    flat = motion_lib.synthetic(model, num_motions=6, num_frames=60, seed=3)
    torch.manual_seed(0)
    task = HumanoidSMPLIM(im_cfg(64, flat), SIM_PARAMS, 1, "cuda", 0, True)
    missing = [n for n in _recorded()["touched"] if not hasattr(task, n)]
    assert not missing, f"the live task lacks attributes the reference's callers touch: {missing}"
    clip_obs, clip_actions = 5.0, 1.0                  # the reference's VecTaskPythonWrapper(task, rl_device, 5.0, 1.0)
    task.reset()
    c = lambda x: x.contiguous()  # noqa: E731
    g = lambda x: x.detach().cpu().numpy()  # noqa: E731
    for i in range(32):
        task.step(torch.clamp(torch.rand(64, 75, device="cuda:0") * 2 - 1, -clip_actions, clip_actions))
        obs = torch.clamp(task.obs_buf, -clip_obs, clip_obs)
        assert bool(torch.isfinite(obs).all() and torch.isfinite(task.rew_buf).all()), f"step {i}"
        assert obs.shape == (64, 461) and "terminate" in task.extras
        rbs = task._rigid_body_state.view(64, -1, 13)
        args = (c(rbs[..., 0:3]), c(rbs[..., 3:7]), task._target_rb_pos, task._target_rb_rot, c(task._dof_pos), c(task._dof_vel),
                task._target_dof_pos, c(rbs[..., 7:10]), c(rbs[..., 10:13]), task._reset_ref_motion_bodies)
        ours = g(task.compute_imitation_obs(*args, True, True))
        ref = R.compute_humanoid_observations_imitation(*(g(a) for a in args), True, True)
        # the port runs in float32 on the CPU with its own operation order: large entries (|x| ~ 20) differ by a few ulp (1.1e-5
        # measured), hence the relative term next to the absolute 1e-5
        np.testing.assert_allclose(ours, ref, rtol=1e-5, atol=1e-5, err_msg=f"step {i}")
        ids = task.reset_buf.nonzero(as_tuple=False).flatten()
        if len(ids):
            task.reset(ids)
