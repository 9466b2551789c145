"""CPU-side checks: C ABI exports, struct layouts, shim cross-checks, model compiler, host logic."""
import ctypes as C
import os
import re
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    from vid2player3d_b200 import build, native
    lib = build.build()
    from vid2player3d_b200 import native_v2p
    from vid2player3d_b200 import ball_gen
    hdr = "".join(open(os.path.join(ROOT, "include", h)).read() for h in ("b200env.h", "b200env_v2p.h", "b200ball.h"))
    declared = sorted(set(re.findall(r"\b(b200(?:env|v2p|ball)_[a-z_0-9]+)\s*\(", hdr)))
    assert declared == sorted(native.SYMBOLS + native_v2p.SYMBOLS + ball_gen.SYMBOLS)
    L = C.CDLL(lib)  # loads without a GPU; no compute call is made here
    for name in declared:
        assert hasattr(L, name), name
    from vid2player3d_b200 import abi
    assert L.b200env_abi_version() == abi.ABI_VERSION


def test_struct_layouts_match_header(tmp_path):
    from vid2player3d_b200 import abi
    src = tmp_path / "sz.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "%s/include/b200env.h"\n'
                   'int main(){printf("%%zu %%zu %%zu %%zu %%zu %%zu\\n",sizeof(b200_model_t),sizeof(b200_cfg_t),'
                   'sizeof(b200_motion_lib_t),sizeof(b200_buffers_t),offsetof(b200_model_t,kp),offsetof(b200_cfg_t,key_body));}' % ROOT)
    exe = tmp_path / "sz"
    subprocess.check_call(["gcc", str(src), "-o", str(exe)])
    got = [int(x) for x in subprocess.check_output([str(exe)]).split()]
    want = [C.sizeof(abi.Model), C.sizeof(abi.Cfg), C.sizeof(abi.MotionLibView), C.sizeof(abi.Buffers), abi.Model.kp.offset,
            abi.Cfg.key_body.offset]
    assert got == want
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "%s/include/b200env_v2p.h"\n'
                   'int main(){printf("%%zu %%zu %%zu %%zu %%zu %%zu %%zu %%zu\\n",sizeof(b200v2p_state_t),sizeof(b200v2p_ctrl_t),'
                   'offsetof(b200v2p_state_t,root_pos),offsetof(b200v2p_ctrl_t,est_x),sizeof(b200v2p_treset_t),sizeof(b200v2p_areset_t),'
                   'offsetof(b200v2p_treset_t,swing_type_cycle),offsetof(b200v2p_areset_t,terminate_buf));}' % ROOT)
    subprocess.check_call(["gcc", str(src), "-o", str(exe)])
    got = [int(x) for x in subprocess.check_output([str(exe)]).split()]
    assert got == [C.sizeof(abi.V2PState), C.sizeof(abi.V2PCtrl), abi.V2PState.root_pos.offset, abi.V2PCtrl.est_x.offset,
                   C.sizeof(abi.V2PTaskReset), C.sizeof(abi.V2PActorReset), abi.V2PTaskReset.swing_type_cycle.offset,
                   abi.V2PActorReset.terminate_buf.offset]


def test_no_gpu_means_loud_failure():
    """the product path has no CPU fallback: creating an env without a CUDA device raises"""
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from vid2player3d_b200 import abi, model_compiler, native
    mod = model_compiler.load_compiled("smpl_mesh_humanoid_amass_v1")
    m, v = abi.pack_model(mod, 1.0)
    with pytest.raises(RuntimeError, match="no CUDA device|CUDA error"):
        native.Env(m, v, abi.make_cfg(mod), 4, 0)
    from vid2player3d_b200.tasks import BaseTask
    with pytest.raises(RuntimeError, match="CUDA device only"):
        BaseTask({"device_type": "cpu", "headless": True, "env": {"numEnvs": 1}})


def test_shim_quaternion_helpers_match_poselib_conventions():
    """the only foreign arithmetic of the oracle (isaacgym.torch_utils) is cross-checked against the reference's own poselib
    definitions (their outputs on seeded inputs, tests/golden/poselib_quat.npz) and against closed forms"""
    import sys
    sys.path.insert(0, os.path.join(ROOT, "vid2player3d_b200", "shim"))
    from isaacgym import torch_utils as IG
    P = {k: torch.from_numpy(v) for k, v in np.load(os.path.join(ROOT, "tests", "golden", "poselib_quat.npz")).items()}
    a, b, v, ang = P["a"], P["b"], P["v"], P["ang"]
    assert torch.allclose(IG.quat_mul(a, b), P["quat_mul"], atol=1e-6)
    assert torch.allclose(IG.quat_conjugate(a), P["quat_conjugate"])
    assert torch.allclose(IG.quat_from_angle_axis(ang, v), P["quat_from_angle_axis"], atol=1e-6)
    assert torch.allclose(IG.quat_rotate(a, v), P["quat_rotate"], atol=1e-5)
    # closed forms
    ident = torch.tensor([[0.0, 0, 0, 1]]).repeat(64, 1)
    assert torch.allclose(IG.quat_mul(a, IG.quat_conjugate(a)), ident, atol=1e-6)
    assert torch.allclose(IG.quat_rotate(a, v).norm(dim=-1), v.norm(dim=-1), atol=1e-5)
    assert torch.allclose(IG.normalize_angle(torch.tensor([3.5, -3.5, 0.1])), torch.tensor([3.5 - 2 * np.pi, 2 * np.pi - 3.5, 0.1]), atol=1e-6)


def test_compiled_models():
    from vid2player3d_b200 import abi, model_compiler
    m = model_compiler.load_compiled("smpl_mesh_humanoid_amass_v1")
    assert len(m["parent"]) == 24 and len(m["kp"]) == 69
    assert m["parent"].tolist() == [-1, 0, 1, 2, 3, 0, 5, 6, 7, 0, 9, 10, 11, 12, 11, 14, 15, 16, 17, 11, 19, 20, 21, 22]
    assert abs(m["mass"].sum() - 102.418) < 0.01  # SURVEY.md 7 sanity value
    f = model_compiler.load_compiled("smpl_mesh_humanoid_federer")
    assert len(f["parent"]) == 25 and f["fixed"][-1] == 1 and str(f["body_names"][-1]) == "Racket"
    assert abs(f["dyn_mass"].sum() - f["mass"].sum()) < 1e-9 and f["dyn_mass"][-1] == 0
    ms, verts = abi.pack_model(f, 1.0)
    assert ms.nb == 25 and ms.vmax % 4 == 0 and verts.shape == (25, ms.vmax, 3)
    # principal inertias positive, triangle inequality
    for I in m["inertia"]:
        w = np.linalg.eigvalsh(I)
        assert w.min() > 0 and w[0] + w[1] >= w[2] * (1 - 1e-9)


def test_hull_faces_of_compiled_models_are_closed_outward_meshes():
    """abi.pack_faces (b200env_set_hull_faces): every body's faces form a closed triangle mesh (Euler: F = 2V' - 4 over the vertices
    used), every hull vertex satisfies every plane, normals point away from the centroid; the body permutation of a left-handed
    asset carries the faces with it"""
    from vid2player3d_b200 import abi, model_compiler
    for name in ("smpl_mesh_humanoid_amass_v1", "smpl_mesh_humanoid_nadal"):
        mod = model_compiler.canonical_racket_last(model_compiler.load_compiled(name))
        ms, verts = abi.pack_model(mod, 1.0)
        planes, tris, ntris, tmax = abi.pack_faces(mod, verts)
        assert planes.shape == (ms.nb, tmax, 4) and tris.shape == (ms.nb, tmax, 4) and tmax <= 255
        for b in range(ms.nb):
            nv, nt = int(ms.nverts[b]), int(ntris[b])
            if nv == 0:
                assert nt == 0                                                   # the welded racket has no hull (prims instead)
                continue
            assert nt >= 4
            T = tris[b, :nt, :3].astype(int)
            assert T.max() < nv
            used = np.unique(T)
            edges = {}
            for t in T:
                for i in range(3):
                    e = (t[i], t[(i + 1) % 3])
                    edges[e] = edges.get(e, 0) + 1
            assert all(c == 1 for c in edges.values()) and all((e[1], e[0]) in edges for e in edges)   # oriented, closed, manifold
            assert nt == 2 * len(used) - 4
            V = verts[b, :nv].astype(np.float64)
            sd = V @ planes[b, :nt, :3].T.astype(np.float64) - planes[b, :nt, 3]
            assert sd.max() < 1e-6
            cen = V[used].mean(0)
            assert ((cen @ planes[b, :nt, :3].T - planes[b, :nt, 3]) < 0).all()
            np.testing.assert_allclose(np.linalg.norm(planes[b, :nt, :3], axis=1), 1.0, atol=1e-6)


def test_left_handed_asset_in_canonical_order():
    """nadal (Racket welded to L_Wrist, body 19) -> right-handed body order; head slab normal = the semi_western grip normal"""
    from vid2player3d_b200 import abi, model_compiler, native_v2p
    raw = model_compiler.load_compiled("smpl_mesh_humanoid_nadal")
    fed = model_compiler.load_compiled("smpl_mesh_humanoid_federer")
    m = model_compiler.canonical_racket_last(raw)
    assert [str(x) for x in m["body_names"]] == [str(x) for x in fed["body_names"]]
    assert int(m["parent"][24]) == 17 and int(fed["parent"][24]) == 22 and int(m["fixed"][24]) == 1
    assert np.isclose(m["mass"].sum(), raw["mass"].sum()) and np.isclose(m["dyn_mass"].sum(), raw["dyn_mass"].sum())
    assert np.array_equal(m["dof_of_body"][:24], fed["dof_of_body"][:24])          # DOF order untouched
    assert model_compiler.canonical_racket_last(fed) is fed
    h = abi.racket_head_from_prims(m)
    x, y, z, w = h["racket_head_quat"]
    normal = np.array([2 * (x * y - z * w), 1 - 2 * (x * x + z * z), 2 * (y * z + x * w)])   # R(q) e_y
    np.testing.assert_allclose(normal, native_v2p.GRIP_NORMAL['semi_western'], atol=1e-12)
    np.testing.assert_allclose(abi.racket_head_from_prims(fed)["racket_head_quat"], (0, 0, 0, 1), atol=1e-12)
    cfg = abi.make_cfg(m, ball={}, task_mode=1, pd_mode=1)
    assert cfg.racket_body == 24 and abs(cfg.racket_head_halfthick - 0.015 * 2 ** 0.5) < 1e-6


def test_model_compiler_reproduces_committed_blob():
    ref = os.path.join(ROOT, "tests", "golden", "amass_asset", "mjcf", "smpl_mesh_humanoid_amass_v1.xml")   # the reference's asset
    from vid2player3d_b200 import model_compiler
    a = model_compiler.compile_mjcf(ref)
    b = model_compiler.load_compiled("smpl_mesh_humanoid_amass_v1")
    for k in ("mass", "com", "inertia", "verts", "kp", "limits", "offset"):
        np.testing.assert_allclose(a[k], b[k], atol=1e-12)


def test_synthetic_motion_lib_is_consistent():
    """FK consistency of the synthetic MoCap buffer: grs/gts follow from lrs and the skeleton"""
    from vid2player3d_b200 import model_compiler, motion_lib
    from oracle import ref_port as R
    m = model_compiler.load_compiled("smpl_mesh_humanoid_amass_v1")
    flat = motion_lib.synthetic(m, num_motions=3, num_frames=20, seed=1, ragged=True)
    assert flat.length_starts.tolist() == [0] + np.cumsum(flat.num_frames)[:-1].tolist()
    assert flat.gts.shape[0] == flat.num_frames.sum()
    np.testing.assert_allclose(np.linalg.norm(flat.grs, axis=-1), 1, atol=1e-6)
    f = 7
    for b in range(1, 24):
        p = m["parent"][b]
        want = R.quat_mul(flat.grs[f, p].astype(np.float64), flat.lrs[f, b].astype(np.float64))
        np.testing.assert_allclose(want, flat.grs[f, b], atol=1e-5)
        np.testing.assert_allclose(flat.gts[f, p] + R.my_quat_rotate(flat.grs[f, p].astype(np.float64), m["offset"][b]),
                                   flat.gts[f, b], atol=1e-5)


def test_physics_oracle_invariants():
    """float64 restatement: momentum drift is O(h) (refining the step shrinks it), weight is carried at rest"""
    from vid2player3d_b200 import abi, model_compiler
    from oracle import physics_ref as P
    mod = model_compiler.load_compiled("smpl_mesh_humanoid_amass_v1")
    rng = np.random.default_rng(0)
    drift = []
    for substeps in (2, 20):
        md = dict(mod); md["armature"] = np.zeros(69)
        m0, verts = abi.pack_model(md, 0.0)
        cfg0 = abi.make_cfg(mod, gravity_z=0.0, ang_damping=0.0, substeps=substeps)
        root = np.zeros((1, 13)); root[:, 2] = 5; root[:, 6] = 1; root[:, 7:10] = [1, 0.5, 0.2]; root[:, 10:13] = [0.5, -1, 2]
        rs = np.random.default_rng(1)
        q = rs.normal(0, 0.3, (1, 69)); qd = rs.normal(0, 2, (1, 69)); tar = np.zeros((1, 69))
        d0 = P.diagnostics(m0, cfg0, root[0], q[0], qd[0])
        P.control_step(m0, verts, cfg0, root, q, qd, tar, n_steps=15)
        d1 = P.diagnostics(m0, cfg0, root[0], q[0], qd[0])
        drift.append(max(np.abs(d1["P"] - d0["P"]).max(), np.abs(d1["L"] - d0["L"]).max()))
    assert drift[1] < 0.2 * drift[0]
    # lying drop (config 1) comes to rest carrying its weight
    m, verts = abi.pack_model(mod, mod["mass"].sum() / 90.0)
    cfg = abi.make_cfg(mod)
    root = np.zeros((1, 13)); root[0, 2] = 0.89; root[0, 6] = 1
    q = np.zeros((1, 69)); qd = np.zeros((1, 69)); tar = np.zeros((1, 69))
    rb, cf = P.control_step(m, verts, cfg, root, q, qd, tar, n_steps=60)
    assert abs(cf[0, :, 2].sum() - mod["mass"].sum() * 9.81) < 2.0
    assert np.abs(qd).max() < 0.05 and abs(root[0, 9]) < 1e-3


def test_vec_task_and_parse_task_surface():
    from vid2player3d_b200.tasks import parse_task as pt
    with pytest.raises(Exception, match="Unrecognized task"):
        class A:  # noqa: D401
            task = "Nope"; device_id = 0; rl_device = "cpu"; physics_engine = 1; device = "cuda"; headless = True
        pt(A, {"env": {}}, {}, None)


def test_reference_config_module_runs_on_the_shim():
    """Level B of the boundary (SURVEY.md 8b): what the reference's own utils/config.py (get_args / load_cfg / parse_sim_params,
    amass_im at 64 envs) hands vid2player3d_b200/shim/isaacgym.  Its inputs to the shim - the custom parameters and command line
    of `gymutil.parse_arguments`, the yaml sim section of `gymutil.parse_sim_config` - and the SimParams fields it ended with were
    recorded from one run of it (tests/golden/make_golden_host.py -> tests/golden/ref_callers.json).  Replayed here in a subprocess
    (sys.modules / sys.argv stay clean): the parsed arguments follow the command line and the parameters' defaults, the Isaac Gym
    defaults the module reads next are set, the sim section lands in SimParams, and every SimParams field the module assigns exists
    on the shim's classes.  The module itself is not part of this repository and is not run."""
    code = r'''
import json, sys
sys.path.insert(0, "%s/vid2player3d_b200/shim")
from isaacgym import gymapi, gymutil
rec = json.load(open("%s/tests/golden/ref_callers.json"))["config"]
pa = rec["parse_arguments"]
types = {"str": str, "int": int, "float": float}
params = [{k: (types[v] if k == "type" else v) for k, v in p.items()} for p in pa["custom_parameters"]]
argv = pa["argv"]
sys.argv = ["run.py"] + argv
args = vars(gymutil.parse_arguments(custom_parameters=params, **pa["kwargs"]))
for p in params:
    dest, flag = p["name"][2:], p.get("action") == "store_true"
    if p["name"] in argv:
        want = True if flag else p["type"](argv[argv.index(p["name"]) + 1])
    else:
        want = p.get("default", False if flag else None)
    assert args[dest] == want, (dest, args[dest], want)
assert args["num_envs"] == 64 and args["headless"] is True and args["cfg"] == "amass_im"
# Isaac Gym's parse_arguments defaults without --sim_device / --pipeline / --flex, read by get_args and parse_sim_params
assert (args["sim_device_type"], args["compute_device_id"], args["use_gpu_pipeline"], args["use_gpu"]) == ("cuda", 0, True, True)
assert args["physics_engine"] == gymapi.SIM_PHYSX and args["slices"] == args["subscenes"] == 0 and args["num_threads"] == 0
sim_cfg = rec["parse_sim_config"]["sim_cfg"]
sp = gymapi.SimParams()
gymutil.parse_sim_config(sim_cfg, sp)
for k, v in sim_cfg.items():
    if k in ("physx", "flex"):
        for kk, vv in v.items():
            assert getattr(getattr(sp, k), kk) == vv, (k, kk)
    else:
        assert getattr(sp, k) == v, k
want = rec["sim_params"]
fresh = gymapi.SimParams()
assert set(want) - {"physx", "flex"} <= set(vars(fresh)), set(want) - set(vars(fresh))
assert set(want["physx"]) <= set(vars(fresh.physx)) and set(want["flex"]) <= set(vars(fresh.flex))
print("OK")
''' % (ROOT, ROOT)
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0 and "OK" in r.stdout, r.stdout[-2000:] + r.stderr[-3000:]


def test_flat_motion_library_file_roundtrip(tmp_path):
    """SURVEY.md 8f-3: the mmap-able on-disk MoCap format holds exactly the arrays the sampler reads"""
    from vid2player3d_b200 import model_compiler, motion_lib
    model = model_compiler.load_compiled("smpl_mesh_humanoid_amass_v1")
    flat = motion_lib.synthetic(model, num_motions=5, num_frames=40, seed=3, ragged=True)
    path = str(tmp_path / "lib.b200ml")
    flat.save_flat(path)
    for mm in (True, False):
        back = motion_lib.FlatMotionLib.load_flat(path, mmap=mm)
        for k in motion_lib.FlatMotionLib.FIELDS:
            a, b = getattr(flat, k), getattr(back, k)
            assert a.dtype == b.dtype and a.shape == b.shape and np.array_equal(a, b), k
    assert isinstance(back.gts, np.ndarray) and motion_lib.FlatMotionLib.load_any(path).num_motions() == 5
    assert os.path.getsize(path) % 64 == 0
    flat.save(str(tmp_path / "lib.npz"))
    assert np.array_equal(motion_lib.FlatMotionLib.load_any(str(tmp_path / "lib.npz")).dvs, flat.dvs)
    (tmp_path / "bad.b200ml").write_bytes(b"not a library" * 4)
    with pytest.raises(ValueError, match="not a B200ML01"):
        motion_lib.FlatMotionLib.load_flat(str(tmp_path / "bad.b200ml"))


def test_quaternion_to_angle_axis_matches_scipy():
    """torch_ops.quaternion_wxyz_to_angle_axis (the ceres formula of konia_transform.py:558-628, test-time `_joint_rot` export)"""
    from scipy.spatial.transform import Rotation
    from vid2player3d_b200.torch_ops import quaternion_wxyz_to_angle_axis
    rng = np.random.default_rng(0)
    q = rng.normal(size=(256, 4))
    q /= np.linalg.norm(q, axis=1, keepdims=True)
    q[0] = [1, 0, 0, 0]
    got = quaternion_wxyz_to_angle_axis(torch.tensor(q)).numpy()
    want = Rotation.from_quat(q[:, [1, 2, 3, 0]]).as_rotvec()
    # q and -q are the same rotation: the formula keeps the angle in (-pi, pi] like the reference
    assert np.abs(got - want).max() < 1e-9
    assert np.all(got[0] == 0)


def test_nn_library_exports_and_layout(tmp_path):
    """libb200nn.so (include/b200nn.h): loads without a GPU, exports every declared symbol, descriptor layout == ctypes mirror,
    and refuses to build a layer without a CUDA device (no fallback)."""
    from vid2player3d_b200 import build, nn
    build.build()
    hdr = open(os.path.join(ROOT, "include", "b200nn.h")).read()
    declared = sorted(set(re.findall(r"\b(b200nn_[a-z_0-9]+)\s*\(", hdr)))
    assert declared == sorted(nn.SYMBOLS)
    L = nn.lib()
    for name in declared:
        assert hasattr(L, name), name
    src = tmp_path / "sz.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "%s/include/b200nn.h"\n'
                   'int main(){printf("%%zu %%zu %%zu\\n",sizeof(b200nn_linear_desc_t),offsetof(b200nn_linear_desc_t,out),'
                   'offsetof(b200nn_linear_desc_t,k_padded));}' % ROOT)
    exe = tmp_path / "sz"
    subprocess.check_call(["gcc", str(src), "-o", str(exe)])
    got = [int(x) for x in subprocess.check_output([str(exe)]).split()]
    assert got == [C.sizeof(nn.LinearDesc), nn.LinearDesc.out.offset, nn.LinearDesc.k_padded.offset]
    if not torch.cuda.is_available():
        with pytest.raises(RuntimeError, match="CUDA device only"):
            nn.Linear(torch.zeros(128, 64, dtype=torch.bfloat16), torch.zeros(8, 64), torch.zeros(8), torch.zeros(128, 64, dtype=torch.bfloat16), 4)


def test_v2p_glue_struct_layouts(tmp_path):
    from vid2player3d_b200 import abi
    src = tmp_path / "sz.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "%s/include/b200env_v2p.h"\n'
                   'int main(){printf("%%zu %%zu %%zu %%zu %%zu %%zu %%zu\\n",sizeof(b200v2p_prestep_t),offsetof(b200v2p_prestep_t,actions),'
                   'sizeof(b200v2p_stream_t),offsetof(b200v2p_stream_t,ring_phase),offsetof(b200v2p_ctrl_t,advance),offsetof(b200v2p_ctrl_t,touch_mask),offsetof(b200v2p_state_t,only_mask));}' % ROOT)
    exe = tmp_path / "sz"
    subprocess.check_call(["gcc", str(src), "-o", str(exe)])
    got = [int(x) for x in subprocess.check_output([str(exe)]).split()]
    assert got == [C.sizeof(abi.V2PPreStep), abi.V2PPreStep.actions.offset, C.sizeof(abi.V2PStream), abi.V2PStream.ring_phase.offset,
                   abi.V2PCtrl.advance.offset, abi.V2PCtrl.touch_mask.offset, abi.V2PState.only_mask.offset]


def test_motion_lib_formats_directory_and_merge(tmp_path):
    """motion_file handling of HumanoidSMPLIM._load_motion (reference humanoid_smpl_im.py:420-440): .npz / .b200ml files, a directory
    of them with motion_file_range, merge = concatenation with rebuilt frame offsets; unknown formats fail loudly"""
    from vid2player3d_b200 import model_compiler, motion_lib as ML
    model = model_compiler.load_compiled("smpl_mesh_humanoid_amass_v1")
    libs = [ML.synthetic(model, num_motions=m, num_frames=20, seed=s, ragged=True) for m, s in ((2, 1), (3, 2), (1, 3))]
    d = tmp_path / "libs"
    d.mkdir()
    for i, l in enumerate(libs):
        l.save_flat(str(d / f"part{i}.b200ml"))
    libs[0].save(str(tmp_path / "one.npz"))
    a = ML.FlatMotionLib.load_any(str(tmp_path / "one.npz"))
    assert np.array_equal(a.gts, libs[0].gts)
    merged = ML.FlatMotionLib.load_any(str(d))
    assert merged.num_motions() == 6 and merged.gts.shape[0] == sum(l.gts.shape[0] for l in libs)
    assert np.array_equal(merged.length_starts, np.concatenate([[0], np.cumsum(merged.num_frames)[:-1]]))
    assert np.array_equal(merged.gts[libs[0].gts.shape[0]:libs[0].gts.shape[0] + libs[1].gts.shape[0]], libs[1].gts)
    part = ML.FlatMotionLib.load_any(str(d), motion_file_range=[1, 3])
    assert part.num_motions() == 4 and np.array_equal(part.motion_lengths, np.concatenate([libs[1].motion_lengths, libs[2].motion_lengths]))
    bad = tmp_path / "x.bin"
    bad.write_bytes(b"not a motion library")
    with pytest.raises(ValueError, match="unknown motion library format"):
        ML.FlatMotionLib.load_any(str(bad))
    with pytest.raises(FileNotFoundError):
        ML.FlatMotionLib.load_any(str(tmp_path / "missing.pth"))
    empty = tmp_path / "empty"
    empty.mkdir()
    with pytest.raises(FileNotFoundError):
        ML.FlatMotionLib.load_any(str(empty))


def test_from_reference_motion_lib_pickle():
    """a reference `torch.save(motion_lib)` pickle (what every reference yaml's motion_file names) loads through
    FlatMotionLib.load_any / from_reference.  The pickle (tests/golden/ref_motion_lib.pth) was written by the reference's
    MotionLib from the synthetic library rebuilt below (tests/golden/make_golden_host.py); it is loaded in a subprocess with a
    stand-in for the reference's `utils.motion_lib.MotionLib` class (unpickling restores the instance attributes only)."""
    code = r'''
import os, sys, types
sys.path.insert(0, %(root)r)
import numpy as np, torch
from vid2player3d_b200 import model_compiler, motion_lib
from vid2player3d_b200.motion_lib import FlatMotionLib
sys.modules["utils"] = types.ModuleType("utils")
sys.modules["utils.motion_lib"] = ml_mod = types.ModuleType("utils.motion_lib")
ml_mod.MotionLib = type("MotionLib", (), {})
model = model_compiler.load_compiled("smpl_mesh_humanoid_amass_v1")
flat = motion_lib.synthetic(model, num_motions=3, num_frames=12, seed=11, sigma=0.08, ragged=True)
flat.min_verts_h = np.linspace(-0.02, 0.03, 3).astype(np.float32)
flat.motion_bodies = np.random.default_rng(5).normal(size=(3, 11)).astype(np.float32)
back = FlatMotionLib.load_any(os.path.join(%(root)r, "tests", "golden", "ref_motion_lib.pth"))
for k in FlatMotionLib.FIELDS:
    assert np.array_equal(np.asarray(getattr(back, k)), np.asarray(getattr(flat, k))), k
print("ok")
''' % {"root": ROOT}
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and r.stdout.strip().endswith("ok"), r.stdout[-1500:] + r.stderr[-2500:]
